// d2pc_mesh.cu -- row m1: a triangle mesh of ONE frame's lattice (the unmasked emit rows, row i = r * C + c of an
// R x C lattice).  Our own spec, frozen in oracle/d2pc_mesh_oracle.py (no reference code; the vertex normals follow
// Open3D's ComputeVertexNormals):
//   valid     keep[i] (when given) and all three coordinates finite
//   quads     q = r (C - 1) + c, corners a (r, c), b (r, c+1), p (r+1, c), d (r+1, c+1); four valid corners: split
//             along the shorter diagonal (a-d on ties) into T0, T1; three: the one triangle of those corners
//   filter    float64: n = (p1 - p0) x (p2 - p0), n.n > 0; s = (p0 + p1) + p2, n.s < 0;
//             (n.s)^2 >= cos2 (n.n) (s.s); optionally every edge's d2 <= max_edge^2
//   output    triangles by quad, T0 before T1; vertices = valid (optionally: referenced) rows in lattice order;
//             vertex normal = sum of the adjacent kept triangles' n in ascending triangle order, normalised
// Every CTA handles one segment of kMeshTile columns of one lattice row (quads or vertices), so tiles in launch
// order are tiles in output order and one scan of the per-tile counts gives every output offset.  No atomics on the
// outputs: the result repeats bit for bit.
//   mesh_classify_kernel  quad code (configuration, which of T0 / T1 survive) + triangles per tile
//   mesh_vflag_kernel     per row: is it a vertex + vertices per tile
//   mesh_scan_kernel      exclusive scan of both tile-count arrays (one CTA each), totals -> the output counts
//   mesh_vertex_kernel    compacted xyz / rgb / row, lattice row -> vertex id map, normals from staged corners
//   mesh_tri_kernel       int32 triangles through the id map
#include <cmath>
#include "d2pc_device.cuh"

namespace d2pc {

constexpr int kMeshTile = 128;           // lattice columns (quads or rows) per CTA, one per thread
constexpr int kMeshStageW = kMeshTile + 2;
constexpr int kMeshScanThreads = 1024;
constexpr int kMeshScanPerThread = 4;
constexpr uint32_t kMeshRemoveUnreferenced = D2PC_MESH_REMOVE_UNREFERENCED, kMeshNormals = D2PC_MESH_NORMALS;

// quad code: bit 0 = T0 kept, bit 1 = T1 kept, bits 2..4 = configuration
enum : uint32_t { kCfgAD = 0, kCfgBP = 1, kCfgNoD = 2, kCfgNoA = 3, kCfgNoB = 4, kCfgNoP = 5 };
// corners a, b, p, d = 0, 1, 2, 3 (row offset = corner >> 1, column offset = corner & 1); the corners of T0 / T1 of
// every configuration, 2 bits each, 6 bits per configuration
constexpr unsigned long long mesh_tri6(int k0, int k1, int k2) { return (unsigned long long)(k0 | k1 << 2 | k2 << 4); }
constexpr unsigned long long kMeshT0 = mesh_tri6(0, 2, 3) | mesh_tri6(0, 2, 1) << 6 | mesh_tri6(0, 2, 1) << 12 |
                                       mesh_tri6(1, 2, 3) << 18 | mesh_tri6(0, 2, 3) << 24 | mesh_tri6(0, 3, 1) << 30;
constexpr unsigned long long kMeshT1 = mesh_tri6(0, 3, 1) | mesh_tri6(1, 2, 3) << 6;   // only a-d / b-p splits
__device__ __forceinline__ uint32_t mesh_corner(uint32_t cfg, int t, int m) {
  return (uint32_t)(((t ? kMeshT1 : kMeshT0) >> (6 * cfg + 2 * m)) & 3ull);
}

struct MeshArgs {
  const float *xyz, *rgb;
  const uint8_t *keep;    // or nullptr
  int32_t R, C;
  int32_t qtpr, vtpr;     // quad / vertex tiles per lattice row
  double cos2, max_edge2;
  int32_t use_edge, remove_unref;
  uint8_t *code;          // [(R-1)(C-1)]
  uint8_t *vflag;         // [R C]
  int32_t *idmap;         // [R C]
  uint32_t *qtile, *vtile;
  float *vxyz, *vrgb;
  int32_t *vrow;
  double *vnormals;
  int32_t *tri;
};

struct D3 { double x, y, z; };

__device__ __forceinline__ D3 mesh_tri_normal(D3 p0, D3 p1, D3 p2) {
  const D3 a{p1.x - p0.x, p1.y - p0.y, p1.z - p0.z}, b{p2.x - p0.x, p2.y - p0.y, p2.z - p0.z};
  return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x};   // Eigen's cross (--fmad=false)
}
__device__ __forceinline__ double mesh_dot(D3 a, D3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ double mesh_d2(D3 q, D3 p) {
  const double dx = q.x - p.x, dy = q.y - p.y, dz = q.z - p.z;
  double d2 = dx * dx;
  d2 += dy * dy;
  d2 += dz * dz;
  return d2;
}

__device__ __forceinline__ bool mesh_tri_keep(D3 p0, D3 p1, D3 p2, const MeshArgs &a) {
  const D3 n = mesh_tri_normal(p0, p1, p2);
  const double nn = mesh_dot(n, n);
  if (!(nn > 0.0)) return false;                          // zero area
  const D3 s{(p0.x + p1.x) + p2.x, (p0.y + p1.y) + p2.y, (p0.z + p1.z) + p2.z};
  const double ns = mesh_dot(n, s);
  if (!(ns < 0.0)) return false;                          // faces away from the camera
  if (!(ns * ns >= a.cos2 * nn * mesh_dot(s, s))) return false;   // grazing: a depth discontinuity
  if (a.use_edge)
    return mesh_d2(p0, p1) <= a.max_edge2 && mesh_d2(p1, p2) <= a.max_edge2 && mesh_d2(p2, p0) <= a.max_edge2;
  return true;
}

__device__ __forceinline__ D3 mesh_pick(const D3 P[4], uint32_t k) {   // constant indices: P stays in registers
  D3 q = P[0];
  if (k == 1) q = P[1];
  if (k == 2) q = P[2];
  if (k == 3) q = P[3];
  return q;
}

__device__ __forceinline__ uint32_t mesh_corner_mask(uint32_t code) {
  const uint32_t cfg = (code >> 2) & 7u;
  uint32_t m = 0;
#pragma unroll
  for (int t = 0; t < 2; ++t)
    if (code & (1u << t))
      m |= (1u << mesh_corner(cfg, t, 0)) | (1u << mesh_corner(cfg, t, 1)) | (1u << mesh_corner(cfg, t, 2));
  return m;
}

// lattice rows r0 .. r0 + NR - 1, columns c0 - 1 .. c0 + kMeshTile, staged once per CTA; outside the lattice = invalid
template <int NR>
struct MeshStage {
  float x[NR][kMeshStageW], y[NR][kMeshStageW], z[NR][kMeshStageW];
  uint8_t v[NR][kMeshStageW];
  __device__ __forceinline__ D3 p(int rr, int cc) const { return {(double)x[rr][cc], (double)y[rr][cc], (double)z[rr][cc]}; }
};

template <int NR>
__device__ __forceinline__ void mesh_stage(MeshStage<NR> &s, const MeshArgs &a, int r0, int c0) {
  for (int e = threadIdx.x; e < NR * kMeshStageW; e += kMeshTile) {
    const int rr = e / kMeshStageW, cc = e - rr * kMeshStageW;
    const int r = r0 + rr, c = c0 - 1 + cc;
    float x = 0.0f, y = 0.0f, z = 0.0f;
    bool ok = false;
    if (r >= 0 && r < a.R && c >= 0 && c < a.C) {
      const size_t i = (size_t)r * (size_t)a.C + (size_t)c;
      x = __ldg(a.xyz + 3 * i);
      y = __ldg(a.xyz + 3 * i + 1);
      z = __ldg(a.xyz + 3 * i + 2);
      ok = (!a.keep || __ldg(a.keep + i) != 0) && isfinite(x) && isfinite(y) && isfinite(z);
    }
    s.x[rr][cc] = x;
    s.y[rr][cc] = y;
    s.z[rr][cc] = z;
    s.v[rr][cc] = ok ? 1 : 0;
  }
  __syncthreads();
}

__device__ __forceinline__ uint32_t mesh_excl_scan(uint32_t v, uint32_t *s_warp, uint32_t *total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  uint32_t incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t y = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += y;
  }
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();
  uint32_t woff = 0, t = 0;
  for (int k = 0; k < nw; ++k) { const uint32_t x = s_warp[k]; if (k < warp) woff += x; t += x; }
  *total = t;
  __syncthreads();
  return woff + incl - v;
}

__global__ void __launch_bounds__(kMeshTile) mesh_classify_kernel(MeshArgs a) {
  __shared__ MeshStage<2> s;
  __shared__ uint32_t s_warp[kMeshTile / 32];
  const int r = (int)blockIdx.x / a.qtpr, c0 = ((int)blockIdx.x - r * a.qtpr) * kMeshTile;
  mesh_stage<2>(s, a, r, c0);
  const int j = threadIdx.x + 1, c = c0 + (int)threadIdx.x;
  uint32_t code = 0;
  if (c < a.C - 1) {
    const bool va = s.v[0][j], vb = s.v[0][j + 1], vp = s.v[1][j], vd = s.v[1][j + 1];
    const int nv = (int)va + (int)vb + (int)vp + (int)vd;
    if (nv >= 3) {
      const D3 P[4] = {s.p(0, j), s.p(0, j + 1), s.p(1, j), s.p(1, j + 1)};
      uint32_t cfg;
      if (nv == 4) cfg = mesh_d2(P[0], P[3]) <= mesh_d2(P[1], P[2]) ? kCfgAD : kCfgBP;
      else cfg = !vd ? kCfgNoD : (!va ? kCfgNoA : (!vb ? kCfgNoB : kCfgNoP));
      code = cfg << 2;
      for (int t = 0; t < (nv == 4 ? 2 : 1); ++t)
        if (mesh_tri_keep(mesh_pick(P, mesh_corner(cfg, t, 0)), mesh_pick(P, mesh_corner(cfg, t, 1)),
                          mesh_pick(P, mesh_corner(cfg, t, 2)), a))
          code |= 1u << t;
    }
    a.code[(size_t)r * (size_t)(a.C - 1) + (size_t)c] = (uint8_t)code;
  }
  uint32_t total;
  mesh_excl_scan((uint32_t)__popc(code & 3u), s_warp, &total);
  if (threadIdx.x == 0) a.qtile[blockIdx.x] = total;
}

// which of the <= 4 quads around row (r, c) use it as a corner of a kept triangle
__device__ __forceinline__ bool mesh_referenced(const MeshArgs &a, int r, int c) {
  const size_t qc = (size_t)(a.C - 1);
  bool used = false;
  if (r >= 1 && c >= 1) used |= (mesh_corner_mask(a.code[(size_t)(r - 1) * qc + (c - 1)]) >> 3) & 1u;   // as d
  if (r >= 1 && c < a.C - 1) used |= (mesh_corner_mask(a.code[(size_t)(r - 1) * qc + c]) >> 2) & 1u;    // as p
  if (r < a.R - 1 && c >= 1) used |= (mesh_corner_mask(a.code[(size_t)r * qc + (c - 1)]) >> 1) & 1u;    // as b
  if (r < a.R - 1 && c < a.C - 1) used |= mesh_corner_mask(a.code[(size_t)r * qc + c]) & 1u;           // as a
  return used;
}

__global__ void __launch_bounds__(kMeshTile) mesh_vflag_kernel(MeshArgs a) {
  __shared__ uint32_t s_warp[kMeshTile / 32];
  const int r = (int)blockIdx.x / a.vtpr, c = ((int)blockIdx.x - r * a.vtpr) * kMeshTile + (int)threadIdx.x;
  uint32_t flag = 0;
  if (c < a.C) {
    const size_t i = (size_t)r * (size_t)a.C + (size_t)c;
    const float x = __ldg(a.xyz + 3 * i), y = __ldg(a.xyz + 3 * i + 1), z = __ldg(a.xyz + 3 * i + 2);
    flag = (!a.keep || __ldg(a.keep + i) != 0) && isfinite(x) && isfinite(y) && isfinite(z);
    if (flag && a.remove_unref) flag = mesh_referenced(a, r, c);
    a.vflag[i] = (uint8_t)flag;
  }
  uint32_t total;
  mesh_excl_scan(flag, s_warp, &total);
  if (threadIdx.x == 0) a.vtile[blockIdx.x] = total;
}

// exclusive scan in place, one CTA per array (0: triangle tiles, 1: vertex tiles); totals -> the output counts
__global__ void __launch_bounds__(kMeshScanThreads) mesh_scan_kernel(uint32_t *qtile, uint32_t nq, uint32_t *tri_count,
                                                                     uint32_t *vtile, uint32_t nv, uint32_t *vtx_count) {
  __shared__ uint32_t s_warp[32];
  __shared__ uint32_t s_carry;
  uint32_t *arr = blockIdx.x == 0 ? qtile : vtile;
  const uint32_t n = blockIdx.x == 0 ? nq : nv;
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  for (uint32_t base = 0; base < n; base += kMeshScanThreads * kMeshScanPerThread) {
    const uint32_t i0 = base + threadIdx.x * kMeshScanPerThread;
    uint32_t v[kMeshScanPerThread], sum = 0;
#pragma unroll
    for (int k = 0; k < kMeshScanPerThread; ++k) { v[k] = i0 + k < n ? arr[i0 + k] : 0u; sum += v[k]; }
    uint32_t total;
    uint32_t ex = s_carry + mesh_excl_scan(sum, s_warp, &total);
#pragma unroll
    for (int k = 0; k < kMeshScanPerThread; ++k) {
      if (i0 + k < n) arr[i0 + k] = ex;
      ex += v[k];
    }
    __syncthreads();
    if (threadIdx.x == 0) s_carry += total;
    __syncthreads();
  }
  if (threadIdx.x == 0) *(blockIdx.x == 0 ? tri_count : vtx_count) = s_carry;
}

template <bool NORMALS>
__global__ void __launch_bounds__(kMeshTile) mesh_vertex_kernel(MeshArgs a) {
  __shared__ MeshStage<NORMALS ? 3 : 1> s;   // rows r - 1 .. r + 1 (only used with normals)
  __shared__ uint32_t s_warp[kMeshTile / 32];
  const int r = (int)blockIdx.x / a.vtpr, c0 = ((int)blockIdx.x - r * a.vtpr) * kMeshTile;
  const int c = c0 + (int)threadIdx.x;
  if (NORMALS) mesh_stage<NORMALS ? 3 : 1>(s, a, r - 1, c0);
  const size_t i = (size_t)r * (size_t)a.C + (size_t)c;
  const uint32_t flag = c < a.C ? a.vflag[i] : 0u;
  uint32_t total;
  const uint32_t v = a.vtile[blockIdx.x] + mesh_excl_scan(flag, s_warp, &total);
  if (!flag) return;
  a.idmap[i] = (int32_t)v;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    a.vxyz[3 * (size_t)v + k] = __ldg(a.xyz + 3 * i + k);
    a.vrgb[3 * (size_t)v + k] = __ldg(a.rgb + 3 * i + k);
  }
  a.vrow[v] = (int32_t)i;
  if (!NORMALS) return;
  // adjacent quads in ascending quad order and this row's corner in each: (r-1, c-1) d, (r-1, c) p, (r, c-1) b, (r, c) a
  D3 acc{0.0, 0.0, 0.0};
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int qr = r - 1 + (k >> 1), qc = c - 1 + (k & 1);
    const uint32_t me = 3 - k;
    if (qr < 0 || qr >= a.R - 1 || qc < 0 || qc >= a.C - 1) continue;
    const uint32_t code = a.code[(size_t)qr * (size_t)(a.C - 1) + (size_t)qc];
    const uint32_t cfg = (code >> 2) & 7u;
    for (int t = 0; t < 2; ++t) {
      if (!(code & (1u << t))) continue;
      const uint32_t k0 = mesh_corner(cfg, t, 0), k1 = mesh_corner(cfg, t, 1), k2 = mesh_corner(cfg, t, 2);
      if (k0 != me && k1 != me && k2 != me) continue;
      const int sr = qr - (r - 1), sc = qc - (c0 - 1);   // staged position of corner a
      const D3 P[3] = {s.p(sr + (k0 >> 1), sc + (k0 & 1)), s.p(sr + (k1 >> 1), sc + (k1 & 1)),
                       s.p(sr + (k2 >> 1), sc + (k2 & 1))};
      const D3 n = mesh_tri_normal(P[0], P[1], P[2]);
      acc = {acc.x + n.x, acc.y + n.y, acc.z + n.z};
    }
  }
  const double ss = mesh_dot(acc, acc);
  D3 nv{0.0, 0.0, 1.0};
  if (ss != 0.0) {
    const double len = sqrt(ss);
    nv = {acc.x / len, acc.y / len, acc.z / len};
  }
  a.vnormals[3 * (size_t)v] = nv.x;
  a.vnormals[3 * (size_t)v + 1] = nv.y;
  a.vnormals[3 * (size_t)v + 2] = nv.z;
}

__global__ void __launch_bounds__(kMeshTile) mesh_tri_kernel(MeshArgs a) {
  __shared__ uint32_t s_warp[kMeshTile / 32];
  const int r = (int)blockIdx.x / a.qtpr, c = ((int)blockIdx.x - r * a.qtpr) * kMeshTile + (int)threadIdx.x;
  const uint32_t code = c < a.C - 1 ? a.code[(size_t)r * (size_t)(a.C - 1) + (size_t)c] : 0u;
  uint32_t total;
  size_t t_out = a.qtile[blockIdx.x] + mesh_excl_scan((uint32_t)__popc(code & 3u), s_warp, &total);
  const uint32_t cfg = (code >> 2) & 7u;
  for (int t = 0; t < 2; ++t) {
    if (!(code & (1u << t))) continue;
#pragma unroll
    for (int m = 0; m < 3; ++m) {
      const uint32_t k = mesh_corner(cfg, t, m);
      a.tri[3 * t_out + m] = a.idmap[(size_t)(r + (k >> 1)) * (size_t)a.C + (size_t)(c + (k & 1))];
    }
    ++t_out;
  }
}

struct MeshLayout {
  size_t code, vflag, idmap, qtile, vtile, total;
  uint32_t qtiles, vtiles;
  int32_t qtpr, vtpr;
};

static MeshLayout mesh_layout(uint32_t rows, uint32_t cols) {
  MeshLayout L;
  L.qtpr = cols >= 2 ? (int32_t)((cols - 2) / kMeshTile + 1) : 0;
  L.vtpr = (int32_t)((cols - 1) / kMeshTile + 1);
  L.qtiles = rows >= 2 ? (rows - 1) * (uint32_t)L.qtpr : 0u;
  L.vtiles = rows * (uint32_t)L.vtpr;
  const size_t n = (size_t)rows * cols, q = rows >= 2 && cols >= 2 ? (size_t)(rows - 1) * (cols - 1) : 0;
  size_t off = 0;
  L.code = off;  off = align_up(off + q, 256);
  L.vflag = off; off = align_up(off + n, 256);
  L.idmap = off; off = align_up(off + n * sizeof(int32_t), 256);
  L.qtile = off; off = align_up(off + (size_t)L.qtiles * sizeof(uint32_t) + 4, 256);
  L.vtile = off; off = align_up(off + (size_t)L.vtiles * sizeof(uint32_t) + 4, 256);
  L.total = off;
  return L;
}

static bool mesh_shape_ok(uint32_t rows, uint32_t cols) {
  return rows >= 1 && cols >= 1 && (unsigned long long)rows * cols < (1ull << 31);
}

}  // namespace d2pc

using namespace d2pc;

extern "C" int d2pc_grid_mesh_scratch_bytes(uint32_t rows, uint32_t cols, size_t *bytes) {
  if (!bytes || !mesh_shape_ok(rows, cols)) return D2PC_ERR_INVALID_ARGUMENT;
  *bytes = mesh_layout(rows, cols).total;
  return D2PC_OK;
}

extern "C" int d2pc_grid_mesh_enqueue(const float *d_xyz, const float *d_rgb, const uint8_t *d_keep, uint32_t rows,
                                      uint32_t cols, double max_edge, double cos2, uint32_t flags, void *d_scratch,
                                      size_t scratch_bytes, float *d_vtx_xyz, float *d_vtx_rgb, int32_t *d_vtx_row,
                                      double *d_vtx_normals, uint32_t *d_vtx_count, int32_t *d_tri,
                                      uint32_t *d_tri_count, void *stream) {
  if (!d_xyz || !d_rgb || !d_scratch || !d_vtx_xyz || !d_vtx_rgb || !d_vtx_row || !d_vtx_count || !d_tri_count)
    return D2PC_ERR_INVALID_ARGUMENT;
  if (!mesh_shape_ok(rows, cols) || (flags & ~(kMeshRemoveUnreferenced | kMeshNormals)) != 0)
    return D2PC_ERR_INVALID_ARGUMENT;
  if ((flags & kMeshNormals) && !d_vtx_normals) return D2PC_ERR_INVALID_ARGUMENT;
  if (rows >= 2 && cols >= 2 && !d_tri) return D2PC_ERR_INVALID_ARGUMENT;
  if (!(cos2 >= 0.0 && cos2 <= 1.0) || max_edge != max_edge || std::isinf(max_edge)) return D2PC_ERR_INVALID_ARGUMENT;
  if (((uintptr_t)d_scratch & 255u) != 0) return D2PC_ERR_INVALID_ARGUMENT;
  const MeshLayout L = mesh_layout(rows, cols);
  if (scratch_bytes < L.total) return D2PC_ERR_WORKSPACE_TOO_SMALL;
  uint8_t *base = (uint8_t *)d_scratch;
  MeshArgs a;
  a.xyz = d_xyz;
  a.rgb = d_rgb;
  a.keep = d_keep;
  a.R = (int32_t)rows;
  a.C = (int32_t)cols;
  a.qtpr = L.qtpr;
  a.vtpr = L.vtpr;
  a.cos2 = cos2;
  a.use_edge = max_edge > 0.0 ? 1 : 0;
  a.max_edge2 = max_edge > 0.0 ? max_edge * max_edge : 0.0;
  a.remove_unref = (flags & kMeshRemoveUnreferenced) ? 1 : 0;
  a.code = base + L.code;
  a.vflag = base + L.vflag;
  a.idmap = (int32_t *)(base + L.idmap);
  a.qtile = (uint32_t *)(base + L.qtile);
  a.vtile = (uint32_t *)(base + L.vtile);
  a.vxyz = d_vtx_xyz;
  a.vrgb = d_vtx_rgb;
  a.vrow = d_vtx_row;
  a.vnormals = d_vtx_normals;
  a.tri = d_tri;
  cudaStream_t st = (cudaStream_t)stream;
  if (L.qtiles > 0) {
    mesh_classify_kernel<<<L.qtiles, kMeshTile, 0, st>>>(a);
    D2PC_CHECK_LAUNCH();
  }
  mesh_vflag_kernel<<<L.vtiles, kMeshTile, 0, st>>>(a);
  D2PC_CHECK_LAUNCH();
  mesh_scan_kernel<<<2, kMeshScanThreads, 0, st>>>(a.qtile, L.qtiles, d_tri_count, a.vtile, L.vtiles, d_vtx_count);
  D2PC_CHECK_LAUNCH();
  if (flags & kMeshNormals) mesh_vertex_kernel<true><<<L.vtiles, kMeshTile, 0, st>>>(a);
  else mesh_vertex_kernel<false><<<L.vtiles, kMeshTile, 0, st>>>(a);
  D2PC_CHECK_LAUNCH();
  if (L.qtiles > 0) {
    mesh_tri_kernel<<<L.qtiles, kMeshTile, 0, st>>>(a);
    D2PC_CHECK_LAUNCH();
  }
  return D2PC_OK;
}
