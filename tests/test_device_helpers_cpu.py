"""CPU: the host plumbing of the device stages (image_to_pointcloud_b200/_device.py) on CPU tensors: error words,
uploads, pointers and the copies back to the host."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from image_to_pointcloud_b200 import _device as D  # noqa: E402
from image_to_pointcloud_b200 import _lib, cluster  # noqa: E402
from image_to_pointcloud_b200.mesh import TriangleMesh  # noqa: E402

TABLE = ((1, "first"), (2, "second"), (8, "fourth"))
CPU = torch.device("cpu")


def test_raise_errors_known_bits_are_value_errors():
    D.raise_errors(0, TABLE, "here")
    with pytest.raises(ValueError, match="^second$"):
        D.raise_errors(2, TABLE, "here")
    with pytest.raises(ValueError, match="^first; second; fourth$"):
        D.raise_errors(11, TABLE, "here")


def test_raise_errors_unknown_bit_is_a_runtime_error():
    for err in (4, 4 | 1, 16):
        with pytest.raises(RuntimeError, match=f"^here: .*error word {err}\\)$"):
            D.raise_errors(err, TABLE, "here")


def test_cluster_error_word_reports_non_finite_rows_alone():
    """A non-finite row also sets the grid bit (it spoils the bounds); only its own message is raised."""
    both = _lib.CLUSTER_ERR_NONFINITE | _lib.CLUSTER_ERR_GRID
    with pytest.raises(ValueError, match="^points must be finite$"):
        cluster._raise_for(both, 0.1)
    with pytest.raises(ValueError, match="^eps 0.1 is too small"):
        cluster._raise_for(_lib.CLUSTER_ERR_GRID, 0.1)
    with pytest.raises(RuntimeError):
        cluster._raise_for(_lib.CLUSTER_ERR_BOUND, 0.1)
    cluster._raise_for(0, 0.1)


def test_upload_casts_numpy_and_reshapes():
    t = D.upload(np.arange(12, dtype=np.int64).reshape(2, 2, 3), torch.int32, 3, CPU)
    assert t.dtype == torch.int32 and tuple(t.shape) == (4, 3) and t.is_contiguous()
    assert t.flatten().tolist() == list(range(12))
    r = D.upload([[1, 2], [3, 4]], torch.int64, 0, CPU)
    assert r.dtype == torch.int64 and r.tolist() == [1, 2, 3, 4]
    x = torch.arange(6, dtype=torch.float32).reshape(3, 2).t()   # not contiguous
    u = D.upload(x, torch.float32, 3, CPU)
    assert tuple(u.shape) == (2, 3) and u.is_contiguous() and torch.equal(u, x.contiguous())


def test_upload_refuses_a_tensor_of_another_dtype():
    with pytest.raises(ValueError, match="expected torch.float32, got torch.float64"):
        D.upload(torch.zeros((2, 3), dtype=torch.float64), torch.float32, 3, CPU)


def test_ptr():
    assert D.ptr(None) is None
    assert D.ptr(torch.empty(0)) is None
    t = torch.zeros(3)
    assert D.ptr(t) == t.data_ptr()


def test_to_host_of_a_mesh_without_normals():
    mesh = TriangleMesh(torch.zeros((2, 3)), torch.ones((2, 3)), torch.zeros((1, 3), dtype=torch.int32), None,
                        torch.arange(2))
    assert D.to_host(mesh, True) is mesh
    host = D.to_host(mesh, False)
    assert isinstance(host, TriangleMesh) and host.vertex_normals is None
    assert all(isinstance(a, np.ndarray) for f, a in zip(host._fields, host) if f != "vertex_normals")
    assert host.triangles.dtype == np.int32 and host.vertex_rows.tolist() == [0, 1]
    parts = D.to_host((torch.zeros(2), None), False)
    assert type(parts) is tuple and isinstance(parts[0], np.ndarray) and parts[1] is None
