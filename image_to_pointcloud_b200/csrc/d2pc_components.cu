// d2pc_components.cu -- row m3: connected components of ONE triangle mesh (Open3D's ClusterConnectedTriangles) and
// the removal of triangles by a mask (Open3D's RemoveTrianglesByMask + RemoveUnreferencedVertices).  Our own
// restatement, frozen in oracle/d2pc_components_oracle.py:
//   connectivity  two triangles are connected when they share an edge (an unordered vertex pair, degenerate edges
//                 included as written); a non-manifold edge connects every triangle on it
//   numbering     clusters in ascending order of their lowest triangle (the order Open3D's BFS assigns them)
//   area          per triangle Open3D's 0.5 |(p0 - p1) x (p0 - p2)| in float64; per cluster a 64-bit fixed-point
//                 sum q_t = rint(a_t s), s = 2^(62 - e_a - e_T) (max a_t < 2^e_a, T <= 2^e_T), area = sum / s
// Launch sequence of d2pc_mesh_components_enqueue (nothing synchronises the host):
//   comp_setup_kernel       header, error word
//   comp_vertex_kernel      finiteness of the vertex coordinates
//   comp_edge_kernel        per triangle: id check; its three edges into an open-addressed table keyed by the edge,
//                           the value lowered to the lowest triangle by atomicMin; area; max area as float64 bits
//   comp_union_kernel       per triangle: unite with the lowest triangle of each of its edges (d2pc_components.h)
//   comp_root_kernel        root of every triangle (= its component's lowest triangle), roots counted per tile
//   tile_scan_kernel        cluster id of every tile's first root, K
//   comp_number_kernel      cluster id of every root; the area scale
//   comp_accum_kernel       label of every triangle; count and fixed-point area per cluster, one atomic per warp run
//   comp_finish_kernel      cluster areas; K published (0 on an error)
// Removal (d2pc_mesh_filter_enqueue): kept triangles flagged per tile and scanned, referenced vertices marked with
// byte stores and scanned, attributes compacted, kept triangles remapped -- all in input order.
// No floating-point atomics: the result repeats bit for bit.
#include <cmath>

#include "d2pc_components.h"
#include "d2pc_device.cuh"
#include "d2pc_scan.cuh"

namespace d2pc {

constexpr int kCompThreads = 256;
constexpr uint32_t kCompMaxTriangles = 1u << 25;   // 2x the 16.6 M triangles of a 4K high lattice mesh
constexpr uint32_t kCompMaxVertices = 1u << 31;    // vertex ids are int32
// error word bits: 1 a triangle id outside [0, V), 2 a non-finite vertex coordinate, 4 a loop bound exhausted
constexpr int32_t kCompErrTriangle = 1, kCompErrNonFinite = 2, kCompErrBound = 4;

struct __align__(256) CompHeader {
  unsigned long long amax_bits;   // max triangle area as float64 bits (non-negative: ordered like the values)
  double scale;                   // s of the fixed-point areas
  uint32_t n_clusters;
};

struct CompArgs {
  const float *xyz;
  const int32_t *tri;
  uint32_t V, T, cap;
  CompHeader *hdr;
  unsigned long long *keys;   // [cap] edge key of every slot
  uint32_t *vals;             // [cap] lowest triangle of every edge
  uint32_t *eslot;            // [T][3] slot of every edge (kCompNone: the triangle takes no part)
  uint32_t *parent;           // [T]
  uint32_t *root;             // [T]
  double *area;               // [T]
  uint32_t *ttile;            // [ttiles + 1]
  unsigned long long *acc;    // [T] fixed-point area of every cluster
  int32_t *err;
  int32_t *label;             // [T] out: cluster of every triangle
  unsigned long long *ncount; // [T] out: triangles of every cluster (int64)
  double *carea;              // [T] out: area of every cluster
  uint32_t *kcount;
};

__device__ __forceinline__ bool comp_load_tri(const int32_t *tri, uint32_t V, uint32_t t, int32_t v[3]) {
#pragma unroll
  for (int k = 0; k < 3; ++k) v[k] = __ldg(tri + 3 * (size_t)t + k);
  return v[0] >= 0 && (uint32_t)v[0] < V && v[1] >= 0 && (uint32_t)v[1] < V && v[2] >= 0 && (uint32_t)v[2] < V;
}

__global__ void comp_setup_kernel(CompArgs a) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  a.hdr->amax_bits = 0ull;
  a.hdr->scale = 0.0;
  a.hdr->n_clusters = 0;
  *a.err = 0;
}

// finiteness of the coordinates of V vertices (one vertex per lane, one atomic per warp)
__global__ void __launch_bounds__(kCompThreads) comp_vertex_kernel(const float *xyz, uint32_t V, int32_t *err) {
  const uint32_t i = blockIdx.x * kCompThreads + threadIdx.x;
  bool bad = false;
  if (i < V) {
    const float x0 = __ldg(xyz + 3 * (size_t)i), x1 = __ldg(xyz + 3 * (size_t)i + 1), x2 = __ldg(xyz + 3 * (size_t)i + 2);
    bad = !(isfinite(x0) && isfinite(x1) && isfinite(x2));
  }
  if (__ballot_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(err, kCompErrNonFinite);
}

__global__ void __launch_bounds__(kCompThreads) comp_edge_kernel(CompArgs a) {
  const uint32_t t = blockIdx.x * kCompThreads + threadIdx.x;
  double ar = 0.0;
  if (t < a.T) {
    int32_t v[3];
    uint32_t *es = a.eslot + 3 * (size_t)t;
    a.parent[t] = t;
    if (!comp_load_tri(a.tri, a.V, t, v)) {
      atomicOr(a.err, kCompErrTriangle);
      es[0] = es[1] = es[2] = kCompNone;
    } else {
      bool failed = false;
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const uint32_t s = comp_edge_insert(a.keys, a.vals, a.cap, comp_edge_key(v[k], v[k == 2 ? 0 : k + 1]), t);
        failed = failed || s == kCompFail;
        es[k] = s == kCompFail ? kCompNone : s;
      }
      if (failed) atomicOr(a.err, kCompErrBound);
      double p[3][3];
#pragma unroll
      for (int k = 0; k < 3; ++k)
#pragma unroll
        for (int c = 0; c < 3; ++c) p[k][c] = (double)__ldg(a.xyz + 3 * (size_t)v[k] + c);
      ar = comp_triangle_area(p);
      if (!isfinite(ar)) ar = 0.0;   // a non-finite vertex: reported by comp_vertex_kernel
    }
    a.area[t] = ar;
  }
  unsigned long long b = (unsigned long long)__double_as_longlong(ar);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) b = max(b, (unsigned long long)__shfl_xor_sync(0xffffffffu, b, o));
  if ((threadIdx.x & 31) == 0 && b) atomicMax(&a.hdr->amax_bits, b);
}

__global__ void __launch_bounds__(kCompThreads) comp_union_kernel(CompArgs a) {
  const uint32_t t = blockIdx.x * kCompThreads + threadIdx.x;
  if (t >= a.T) return;
  bool failed = false;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const uint32_t s = a.eslot[3 * (size_t)t + k];
    if (s == kCompNone) continue;
    const uint32_t r = a.vals[s];   // <= t, written by the previous launch
    if (r != t) failed = failed || comp_unite(a.parent, t, r, a.T) == kCompFail;
  }
  if (failed) atomicOr(a.err, kCompErrBound);
}

__global__ void __launch_bounds__(kCompThreads) comp_root_kernel(CompArgs a) {
  const uint32_t t = blockIdx.x * kCompThreads + threadIdx.x;
  bool is_root = false;
  if (t < a.T) {
    uint32_t r = comp_find(a.parent, t, a.T);
    if (r == kCompFail) {
      atomicOr(a.err, kCompErrBound);
      r = t;
    }
    a.root[t] = r;
    is_root = r == t;
  }
  const uint32_t n = __syncthreads_count(is_root);
  if (threadIdx.x == 0) a.ttile[blockIdx.x] = n;
}

__global__ void __launch_bounds__(kCompThreads) comp_number_kernel(CompArgs a) {
  __shared__ uint32_t s_warp[kCompThreads / 32];
  const uint32_t t = blockIdx.x * kCompThreads + threadIdx.x;
  const bool is_root = t < a.T && a.root[t] == t;
  uint32_t total;
  const uint32_t id = a.ttile[blockIdx.x] + tile_excl_scan(is_root ? 1u : 0u, s_warp, &total);
  if (is_root) a.label[t] = (int32_t)id;
  if (t == 0) a.hdr->scale = comp_area_scale(__longlong_as_double((long long)a.hdr->amax_bits), a.T);
}

__global__ void __launch_bounds__(kCompThreads) comp_accum_kernel(CompArgs a) {
  const uint32_t t = blockIdx.x * kCompThreads + threadIdx.x;
  const int lane = threadIdx.x & 31;
  uint32_t cid = kCompNone;
  unsigned long long q = 0ull, n = 0ull;
  if (t < a.T) {
    const uint32_t r = a.root[t];
    const int32_t l = a.label[r];   // the root's label, written by the previous launch
    if (r != t) a.label[t] = l;
    cid = (uint32_t)l;
    q = (unsigned long long)__double2ll_rn(a.area[t] * a.hdr->scale);
    n = 1ull;
  }
  // merge each run of equal clusters in the warp (consecutive triangles of a lattice mesh), then one atomic per run
  const uint32_t left = __shfl_up_sync(0xffffffffu, cid, 1);
  const bool head = lane == 0 || left != cid;
  const unsigned heads = __ballot_sync(0xffffffffu, head);
  const int start = 31 - __clz(heads & (0xffffffffu >> (31 - lane)));
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const unsigned long long yq = __shfl_down_sync(0xffffffffu, q, d), yn = __shfl_down_sync(0xffffffffu, n, d);
    const int ys = __shfl_down_sync(0xffffffffu, start, d);
    if (lane + d < 32 && ys == start) { q += yq; n += yn; }
  }
  if (head && cid != kCompNone) {
    atomicAdd(a.ncount + cid, n);
    atomicAdd(a.acc + cid, q);
  }
}

__global__ void __launch_bounds__(kCompThreads) comp_finish_kernel(CompArgs a) {
  const uint32_t c = blockIdx.x * kCompThreads + threadIdx.x;
  if (c >= a.hdr->n_clusters) return;
  a.carea[c] = (double)(long long)a.acc[c] / a.hdr->scale;   // one rounding: the scale is a power of two
}

// publishes K; an error leaves none
__global__ void comp_done_kernel(const int32_t *err, const CompHeader *hdr, uint32_t *kcount) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  *kcount = *err != 0 ? 0u : hdr->n_clusters;
}

__global__ void comp_empty_kernel(int32_t *err, uint32_t T, uint32_t *count_a, uint32_t *count_b) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  *err = T > 0 ? kCompErrTriangle : 0;   // with no vertices every triangle id is out of range
  *count_a = 0;
  if (count_b) *count_b = 0;
}

struct CompLayout {
  size_t hdr, keys, vals, eslot, parent, root, area, ttile, acc, total;
  uint32_t cap, ttiles;
};

static CompLayout comp_layout(uint32_t T) {
  CompLayout L;
  // at most 3T distinct edges: a load factor of at most 3/4, 3/8 for a lattice mesh (about 1.5 T edges)
  const unsigned long long c = 4ull * T;
  L.cap = (uint32_t)(c < 1024ull ? 1024ull : c);
  L.ttiles = (T + kCompThreads - 1) / kCompThreads;
  size_t off = 0;
  L.hdr = off;    off = align_up(off + sizeof(CompHeader), 256);
  L.keys = off;   off = align_up(off + (size_t)L.cap * 8, 256);
  L.vals = off;   off = align_up(off + (size_t)L.cap * 4, 256);
  L.eslot = off;  off = align_up(off + (size_t)T * 12, 256);
  L.parent = off; off = align_up(off + (size_t)T * 4, 256);
  L.root = off;   off = align_up(off + (size_t)T * 4, 256);
  L.area = off;   off = align_up(off + (size_t)T * 8, 256);
  L.ttile = off;  off = align_up(off + ((size_t)L.ttiles + 1) * 4, 256);
  L.acc = off;    off = align_up(off + (size_t)T * 8, 256);
  L.total = off;
  return L;
}

static bool comp_sizes_ok(uint32_t V, uint32_t T) { return V <= kCompMaxVertices && T <= kCompMaxTriangles; }

// ---------------------------------------------------------------------------------------------------------------
// removal by mask
// ---------------------------------------------------------------------------------------------------------------
struct FiltArgs {
  const float *xyz, *rgb;
  const double *nrm;          // or nullptr
  const long long *row;
  const int32_t *tri;
  const uint8_t *keep;
  uint32_t V, T;
  uint8_t *ref;               // [V] 1: the vertex stays
  uint32_t *vtile, *ttile;    // [tiles + 1]
  uint32_t *vmap;             // [V] new id of every vertex that stays
  uint32_t *counts;           // [2] vertices, triangles (scan totals)
  int32_t *err;
  float *oxyz, *orgb;
  double *onrm;
  long long *orow;
  int32_t *otri;
  uint32_t *vcount, *tcount;
  bool unref;
};

__global__ void filt_setup_kernel(FiltArgs a) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  a.counts[0] = a.counts[1] = 0;
  *a.err = 0;
}

__device__ __forceinline__ bool filt_kept(const FiltArgs &a, uint32_t t, int32_t v[3]) {
  if (t >= a.T) return false;
  const bool ok = comp_load_tri(a.tri, a.V, t, v);
  return ok && a.keep[t] != 0;
}

__global__ void __launch_bounds__(kCompThreads) filt_tri_kernel(FiltArgs a) {
  const uint32_t t = blockIdx.x * kCompThreads + threadIdx.x;
  int32_t v[3];
  bool kept = false;
  if (t < a.T) {
    if (!comp_load_tri(a.tri, a.V, t, v)) {
      atomicOr(a.err, kCompErrTriangle);
    } else if (a.keep[t] != 0) {
      kept = true;
      if (a.unref) { a.ref[v[0]] = 1; a.ref[v[1]] = 1; a.ref[v[2]] = 1; }
    }
  }
  const uint32_t n = __syncthreads_count(kept);
  if (threadIdx.x == 0) a.ttile[blockIdx.x] = n;
}

__global__ void __launch_bounds__(kCompThreads) filt_vtx_kernel(FiltArgs a) {
  const uint32_t i = blockIdx.x * kCompThreads + threadIdx.x;
  bool bad = false, stays = false;
  if (i < a.V) {
    const float x0 = __ldg(a.xyz + 3 * (size_t)i), x1 = __ldg(a.xyz + 3 * (size_t)i + 1), x2 = __ldg(a.xyz + 3 * (size_t)i + 2);
    bad = !(isfinite(x0) && isfinite(x1) && isfinite(x2));
    stays = a.ref[i] != 0;
  }
  if (__ballot_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(a.err, kCompErrNonFinite);
  const uint32_t n = __syncthreads_count(stays);
  if (threadIdx.x == 0) a.vtile[blockIdx.x] = n;
}

__global__ void __launch_bounds__(kCompThreads) filt_vtx_write_kernel(FiltArgs a) {
  __shared__ uint32_t s_warp[kCompThreads / 32];
  const uint32_t i = blockIdx.x * kCompThreads + threadIdx.x;
  const bool stays = i < a.V && a.ref[i] != 0;
  uint32_t total;
  const uint32_t j = a.vtile[blockIdx.x] + tile_excl_scan(stays ? 1u : 0u, s_warp, &total);
  if (i >= a.V) return;
  a.vmap[i] = stays ? j : kCompNone;
  if (!stays) return;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    a.oxyz[3 * (size_t)j + k] = __ldg(a.xyz + 3 * (size_t)i + k);
    a.orgb[3 * (size_t)j + k] = __ldg(a.rgb + 3 * (size_t)i + k);
    if (a.nrm) a.onrm[3 * (size_t)j + k] = __ldg(a.nrm + 3 * (size_t)i + k);
  }
  a.orow[j] = __ldg(a.row + i);
}

__global__ void __launch_bounds__(kCompThreads) filt_tri_write_kernel(FiltArgs a) {
  __shared__ uint32_t s_warp[kCompThreads / 32];
  const uint32_t t = blockIdx.x * kCompThreads + threadIdx.x;
  int32_t v[3];
  const bool kept = filt_kept(a, t, v);
  uint32_t total;
  const uint32_t j = a.ttile[blockIdx.x] + tile_excl_scan(kept ? 1u : 0u, s_warp, &total);
  if (!kept) return;
#pragma unroll
  for (int k = 0; k < 3; ++k) a.otri[3 * (size_t)j + k] = (int32_t)a.vmap[v[k]];   // a kept triangle's vertices stay
}

__global__ void filt_done_kernel(FiltArgs a) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const bool bad = *a.err != 0;
  *a.vcount = bad ? 0u : a.counts[0];
  *a.tcount = bad ? 0u : a.counts[1];
}

struct FiltLayout {
  size_t ref, vtile, ttile, vmap, counts, total;
  uint32_t vtiles, ttiles;
};

static FiltLayout filt_layout(uint32_t V, uint32_t T) {
  FiltLayout L;
  L.vtiles = (uint32_t)(((unsigned long long)V + kCompThreads - 1) / kCompThreads);
  L.ttiles = (T + kCompThreads - 1) / kCompThreads;
  size_t off = 0;
  L.counts = off; off = align_up(off + 2 * sizeof(uint32_t), 256);
  L.ref = off;    off = align_up(off + (size_t)V, 256);
  L.vtile = off;  off = align_up(off + ((size_t)L.vtiles + 1) * 4, 256);
  L.ttile = off;  off = align_up(off + ((size_t)L.ttiles + 1) * 4, 256);
  L.vmap = off;   off = align_up(off + (size_t)V * 4, 256);
  L.total = off;
  return L;
}

}  // namespace d2pc

using namespace d2pc;

extern "C" int d2pc_mesh_components_scratch_bytes(uint32_t vertices, uint32_t triangles, size_t *bytes) {
  if (!bytes) return D2PC_ERR_INVALID_ARGUMENT;
  if (!comp_sizes_ok(vertices, triangles)) return D2PC_ERR_UNSUPPORTED;
  *bytes = comp_layout(triangles).total;
  return D2PC_OK;
}

extern "C" int d2pc_mesh_components_enqueue(const float *d_vtx_xyz, uint32_t vertices, const int32_t *d_tri,
                                            uint32_t triangles, void *d_scratch, size_t scratch_bytes,
                                            int32_t *d_out_tri_cluster, int64_t *d_out_cluster_n,
                                            double *d_out_cluster_area, uint32_t *d_out_cluster_count,
                                            int32_t *d_error, void *stream) {
  if (!d_scratch || !d_out_cluster_count || !d_error) return D2PC_ERR_INVALID_ARGUMENT;
  if (vertices > 0 && !d_vtx_xyz) return D2PC_ERR_INVALID_ARGUMENT;
  if (triangles > 0 && (!d_tri || !d_out_tri_cluster || !d_out_cluster_n || !d_out_cluster_area))
    return D2PC_ERR_INVALID_ARGUMENT;
  if (((uintptr_t)d_scratch & 255u) != 0) return D2PC_ERR_INVALID_ARGUMENT;
  if (!comp_sizes_ok(vertices, triangles)) return D2PC_ERR_UNSUPPORTED;
  const CompLayout L = comp_layout(triangles);
  if (scratch_bytes < L.total) return D2PC_ERR_WORKSPACE_TOO_SMALL;
  cudaStream_t st = (cudaStream_t)stream;
  if (vertices == 0 || triangles == 0) {
    comp_empty_kernel<<<1, 32, 0, st>>>(d_error, triangles, d_out_cluster_count, nullptr);
    D2PC_CHECK_LAUNCH();
    if (vertices > 0) {
      comp_vertex_kernel<<<(vertices + kCompThreads - 1) / kCompThreads, kCompThreads, 0, st>>>(d_vtx_xyz, vertices,
                                                                                                 d_error);
      D2PC_CHECK_LAUNCH();
    }
    return D2PC_OK;
  }
  uint8_t *base = (uint8_t *)d_scratch;
  CompArgs a;
  a.xyz = d_vtx_xyz;
  a.tri = d_tri;
  a.V = vertices;
  a.T = triangles;
  a.cap = L.cap;
  a.hdr = (CompHeader *)(base + L.hdr);
  a.keys = (unsigned long long *)(base + L.keys);
  a.vals = (uint32_t *)(base + L.vals);
  a.eslot = (uint32_t *)(base + L.eslot);
  a.parent = (uint32_t *)(base + L.parent);
  a.root = (uint32_t *)(base + L.root);
  a.area = (double *)(base + L.area);
  a.ttile = (uint32_t *)(base + L.ttile);
  a.acc = (unsigned long long *)(base + L.acc);
  a.err = d_error;
  a.label = d_out_tri_cluster;
  a.ncount = (unsigned long long *)d_out_cluster_n;
  a.carea = d_out_cluster_area;
  a.kcount = d_out_cluster_count;
  cudaError_t e = cudaMemsetAsync(a.keys, 0xFF, (size_t)L.cap * 8, st);
  if (e == cudaSuccess) e = cudaMemsetAsync(a.vals, 0xFF, (size_t)L.cap * 4, st);
  if (e == cudaSuccess) e = cudaMemsetAsync(a.acc, 0, (size_t)triangles * 8, st);
  if (e == cudaSuccess) e = cudaMemsetAsync(d_out_cluster_n, 0, (size_t)triangles * 8, st);
  if (e != cudaSuccess) return record_cuda_error(e);
  const uint32_t vt = (uint32_t)(((unsigned long long)vertices + kCompThreads - 1) / kCompThreads);
  comp_setup_kernel<<<1, 32, 0, st>>>(a);
  D2PC_CHECK_LAUNCH();
  comp_vertex_kernel<<<vt, kCompThreads, 0, st>>>(d_vtx_xyz, vertices, d_error);
  D2PC_CHECK_LAUNCH();
  comp_edge_kernel<<<L.ttiles, kCompThreads, 0, st>>>(a);
  D2PC_CHECK_LAUNCH();
  comp_union_kernel<<<L.ttiles, kCompThreads, 0, st>>>(a);
  D2PC_CHECK_LAUNCH();
  comp_root_kernel<<<L.ttiles, kCompThreads, 0, st>>>(a);
  D2PC_CHECK_LAUNCH();
  tile_scan_kernel<<<1, kTileScanThreads, 0, st>>>(a.ttile, L.ttiles, &a.hdr->n_clusters);
  D2PC_CHECK_LAUNCH();
  comp_number_kernel<<<L.ttiles, kCompThreads, 0, st>>>(a);
  D2PC_CHECK_LAUNCH();
  comp_accum_kernel<<<L.ttiles, kCompThreads, 0, st>>>(a);
  D2PC_CHECK_LAUNCH();
  comp_finish_kernel<<<L.ttiles, kCompThreads, 0, st>>>(a);
  D2PC_CHECK_LAUNCH();
  comp_done_kernel<<<1, 32, 0, st>>>(d_error, a.hdr, d_out_cluster_count);
  D2PC_CHECK_LAUNCH();
  return D2PC_OK;
}

extern "C" int d2pc_mesh_filter_scratch_bytes(uint32_t vertices, uint32_t triangles, size_t *bytes) {
  if (!bytes) return D2PC_ERR_INVALID_ARGUMENT;
  if (!comp_sizes_ok(vertices, triangles)) return D2PC_ERR_UNSUPPORTED;
  *bytes = filt_layout(vertices, triangles).total;
  return D2PC_OK;
}

extern "C" int d2pc_mesh_filter_enqueue(const float *d_vtx_xyz, const float *d_vtx_rgb, const double *d_vtx_normals,
                                        const int64_t *d_vtx_row, uint32_t vertices, const int32_t *d_tri,
                                        uint32_t triangles, const uint8_t *d_tri_keep, uint32_t flags,
                                        void *d_scratch, size_t scratch_bytes, float *d_out_xyz, float *d_out_rgb,
                                        double *d_out_normals, int64_t *d_out_row, uint32_t *d_out_vtx_count,
                                        int32_t *d_out_tri, uint32_t *d_out_tri_count, int32_t *d_error,
                                        void *stream) {
  if ((flags & ~(uint32_t)(D2PC_MESH_REMOVE_UNREFERENCED | D2PC_MESH_NORMALS)) != 0) return D2PC_ERR_INVALID_ARGUMENT;
  if (!d_scratch || !d_out_vtx_count || !d_out_tri_count || !d_error) return D2PC_ERR_INVALID_ARGUMENT;
  if (vertices > 0 && (!d_vtx_xyz || !d_vtx_rgb || !d_vtx_row || !d_out_xyz || !d_out_rgb || !d_out_row))
    return D2PC_ERR_INVALID_ARGUMENT;
  if ((flags & D2PC_MESH_NORMALS) && vertices > 0 && (!d_vtx_normals || !d_out_normals))
    return D2PC_ERR_INVALID_ARGUMENT;
  if (triangles > 0 && (!d_tri || !d_tri_keep || !d_out_tri)) return D2PC_ERR_INVALID_ARGUMENT;
  if (((uintptr_t)d_scratch & 255u) != 0) return D2PC_ERR_INVALID_ARGUMENT;
  if (!comp_sizes_ok(vertices, triangles)) return D2PC_ERR_UNSUPPORTED;
  const FiltLayout L = filt_layout(vertices, triangles);
  if (scratch_bytes < L.total) return D2PC_ERR_WORKSPACE_TOO_SMALL;
  cudaStream_t st = (cudaStream_t)stream;
  if (vertices == 0) {
    comp_empty_kernel<<<1, 32, 0, st>>>(d_error, triangles, d_out_vtx_count, d_out_tri_count);
    D2PC_CHECK_LAUNCH();
    return D2PC_OK;
  }
  uint8_t *base = (uint8_t *)d_scratch;
  FiltArgs a;
  a.xyz = d_vtx_xyz;
  a.rgb = d_vtx_rgb;
  a.nrm = (flags & D2PC_MESH_NORMALS) ? d_vtx_normals : nullptr;
  a.row = (const long long *)d_vtx_row;
  a.tri = d_tri;
  a.keep = d_tri_keep;
  a.V = vertices;
  a.T = triangles;
  a.ref = base + L.ref;
  a.vtile = (uint32_t *)(base + L.vtile);
  a.ttile = (uint32_t *)(base + L.ttile);
  a.vmap = (uint32_t *)(base + L.vmap);
  a.counts = (uint32_t *)(base + L.counts);
  a.err = d_error;
  a.oxyz = d_out_xyz;
  a.orgb = d_out_rgb;
  a.onrm = d_out_normals;
  a.orow = (long long *)d_out_row;
  a.otri = d_out_tri;
  a.vcount = d_out_vtx_count;
  a.tcount = d_out_tri_count;
  a.unref = (flags & D2PC_MESH_REMOVE_UNREFERENCED) != 0;
  cudaError_t e = cudaMemsetAsync(a.ref, a.unref ? 0 : 1, (size_t)vertices, st);
  if (e != cudaSuccess) return record_cuda_error(e);
  filt_setup_kernel<<<1, 32, 0, st>>>(a);
  D2PC_CHECK_LAUNCH();
  if (triangles > 0) {
    filt_tri_kernel<<<L.ttiles, kCompThreads, 0, st>>>(a);
    D2PC_CHECK_LAUNCH();
    tile_scan_kernel<<<1, kTileScanThreads, 0, st>>>(a.ttile, L.ttiles, a.counts + 1);
    D2PC_CHECK_LAUNCH();
  }
  filt_vtx_kernel<<<L.vtiles, kCompThreads, 0, st>>>(a);
  D2PC_CHECK_LAUNCH();
  tile_scan_kernel<<<1, kTileScanThreads, 0, st>>>(a.vtile, L.vtiles, a.counts);
  D2PC_CHECK_LAUNCH();
  filt_vtx_write_kernel<<<L.vtiles, kCompThreads, 0, st>>>(a);
  D2PC_CHECK_LAUNCH();
  if (triangles > 0) {
    filt_tri_write_kernel<<<L.ttiles, kCompThreads, 0, st>>>(a);
    D2PC_CHECK_LAUNCH();
  }
  filt_done_kernel<<<1, 32, 0, st>>>(a);
  D2PC_CHECK_LAUNCH();
  return D2PC_OK;
}
