// d2pc_smooth.cu -- row m4: smoothing of ONE triangle mesh (Open3D's FilterSmoothSimple / FilterSmoothLaplacian /
// FilterSmoothTaubin) and the vertex normals of any mesh (m1's rule).  Our restatement, frozen in
// oracle/d2pc_smooth_oracle.py; the per-vertex arithmetic lives in d2pc_smooth.h.
// Launch sequence of d2pc_mesh_smooth_enqueue (nothing synchronises the host):
//   sm_check_kernel        triangle ids and finiteness, before any id indexes anything
//   sm_edge_kernel         per triangle: its three edges into m3's open-addressed edge table (d2pc_components.h)
//   CSR build              per table slot {a, b}: the entries a->b and b->a ({a, a}: one) counted per vertex,
//                          offsets by a tile scan (d2pc_scan.cuh), entries scattered, every segment sorted
//                          (own thread up to kSmSortThread entries, one CTA in shared memory up to kSmSortCta,
//                          one CTA in global memory above)
//   sm_pass_kernel         one launch per pass (two per Taubin iteration), one thread per vertex in input order;
//                          float64 state ping-pongs between two scratch buffers, the first pass reads the inputs
//                          and the last writes the outputs
// d2pc_mesh_vertex_normals_enqueue: sm_check_kernel, the same CSR build over the 3T (vertex, triangle) corners
// (duplicates kept), sm_tri_normal_kernel (each triangle's normal once), sm_vertex_normal_kernel.
// An error makes every later kernel a no-op; every loop has a bound known at launch; no floating-point atomics, so
// the result repeats bit for bit.
#include <cmath>

#include "d2pc_components.h"
#include "d2pc_device.cuh"
#include "d2pc_scan.cuh"
#include "d2pc_smooth.h"

namespace d2pc {

constexpr int kSmThreads = 256;
constexpr uint32_t kSmSortThread = 32;     // a segment this short is insertion-sorted by its own thread
constexpr uint32_t kSmSortCta = 4096;      // up to this: block_bitonic_sort in shared memory (16 KB)
constexpr int kSmSortCtaThreads = 512;
constexpr uint32_t kSmLongCtas = 1024, kSmHugeCtas = 148;
constexpr uint32_t kSmMaxTriangles = 1u << 25;   // m3's limits
constexpr uint32_t kSmMaxVertices = 1u << 31;
// error word bits as m3's: 1 a triangle id outside [0, V), 2 a non-finite value, 4 a loop bound exhausted
constexpr int32_t kSmErrTriangle = 1, kSmErrNonFinite = 2, kSmErrBound = 4;

struct __align__(256) SmHeader {
  uint32_t n_entries, n_long, n_huge;
};

// one CSR (offsets, entries) over the V vertices
struct SmCsr {
  uint32_t V, emax;
  uint32_t *off;     // [V + 1]
  uint32_t *cur;     // [V] degree, then the scatter cursor
  uint32_t *vtile;   // [vtiles + 1]
  uint32_t *ent;     // [emax]
  uint32_t *lst;     // [lcap] long segments, then [hcap] very long ones
  uint32_t lcap, hcap;
  SmHeader *hdr;
  const int32_t *err;
};

// the pairs (vertex, value) a CSR is built from: a table slot {a, b} gives (a, b) and (b, a), {a, a} gives (a, a)
struct SmEdgeSource {
  const unsigned long long *keys;
  uint32_t n;   // table capacity
  __device__ __forceinline__ uint32_t pairs(uint32_t i, uint32_t v[2], uint32_t x[2]) const {
    const unsigned long long k = keys[i];
    if (k == kCompNoKey) return 0;
    const uint32_t lo = (uint32_t)(k >> 32), hi = (uint32_t)k;
    v[0] = lo; x[0] = hi; v[1] = hi; x[1] = lo;
    return lo == hi ? 1u : 2u;
  }
};
// ... and corner k of triangle t gives (tri[t][k], t), duplicates kept
struct SmCornerSource {
  const int32_t *tri;
  uint32_t n;   // 3T
  __device__ __forceinline__ uint32_t pairs(uint32_t i, uint32_t v[2], uint32_t x[2]) const {
    v[0] = (uint32_t)__ldg(tri + i);
    x[0] = i / 3u;
    return 1u;
  }
};

__device__ __forceinline__ bool sm_finite3(const float *p, size_t i) {
  return isfinite(__ldg(p + 3 * i)) && isfinite(__ldg(p + 3 * i + 1)) && isfinite(__ldg(p + 3 * i + 2));
}
__device__ __forceinline__ bool sm_finite3(const double *p, size_t i) {
  return isfinite(__ldg(p + 3 * i)) && isfinite(__ldg(p + 3 * i + 1)) && isfinite(__ldg(p + 3 * i + 2));
}

// thread i checks vertex i (its coordinates, and its colour / normal when given) and triangle i
__global__ void __launch_bounds__(kSmThreads) sm_check_kernel(const float *xyz, const float *rgb, const double *nrm,
                                                              uint32_t V, const int32_t *tri, uint32_t T,
                                                              int32_t *err) {
  const uint32_t i = blockIdx.x * kSmThreads + threadIdx.x;
  int32_t bits = 0;
  if (i < V) {
    bool ok = sm_finite3(xyz, i);
    if (rgb) ok = ok && sm_finite3(rgb, i);
    if (nrm) ok = ok && sm_finite3(nrm, i);
    if (!ok) bits |= kSmErrNonFinite;
  }
  if (i < T) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const int32_t v = __ldg(tri + 3 * (size_t)i + k);
      if (v < 0 || (uint32_t)v >= V) bits |= kSmErrTriangle;
    }
  }
  if (bits) atomicOr(err, bits);
}

__global__ void __launch_bounds__(kSmThreads) sm_edge_kernel(const int32_t *tri, uint32_t T, unsigned long long *keys,
                                                             uint32_t *vals, uint32_t cap, int32_t *err) {
  const uint32_t t = blockIdx.x * kSmThreads + threadIdx.x;
  if (t >= T || *err) return;
  int32_t v[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) v[k] = __ldg(tri + 3 * (size_t)t + k);
  bool failed = false;
#pragma unroll
  for (int k = 0; k < 3; ++k)
    failed = failed || comp_edge_insert(keys, vals, cap, comp_edge_key(v[k], v[k == 2 ? 0 : k + 1]), t) == kCompFail;
  if (failed) atomicOr(err, kSmErrBound);
}

// SCATTER = false: count the pairs of every vertex into cur; true: place each value at its vertex's cursor
template <bool SCATTER, class Source>
__global__ void __launch_bounds__(kSmThreads) sm_csr_fill_kernel(Source src, SmCsr c, int32_t *err) {
  const uint32_t i = blockIdx.x * kSmThreads + threadIdx.x;
  if (i >= src.n || *err) return;
  uint32_t v[2], x[2];
  const uint32_t n = src.pairs(i, v, x);
  for (uint32_t k = 0; k < n; ++k) {
    const uint32_t pos = atomicAdd(c.cur + v[k], 1u);
    if (!SCATTER) continue;
    if (pos < c.emax) c.ent[pos] = x[k];
    else atomicOr(err, kSmErrBound);
  }
}

// per tile of vertices: the sum of the degrees
__global__ void __launch_bounds__(kSmThreads) sm_csr_tile_kernel(SmCsr c) {
  __shared__ uint32_t s_warp[kSmThreads / 32];
  const uint32_t i = blockIdx.x * kSmThreads + threadIdx.x;
  uint32_t total;
  tile_excl_scan(i < c.V ? c.cur[i] : 0u, s_warp, &total);
  if (threadIdx.x == 0) c.vtile[blockIdx.x] = total;
}

// offsets from the scanned tile sums; the cursors start at the offsets
__global__ void __launch_bounds__(kSmThreads) sm_csr_offset_kernel(SmCsr c) {
  __shared__ uint32_t s_warp[kSmThreads / 32];
  const uint32_t i = blockIdx.x * kSmThreads + threadIdx.x;
  const uint32_t d = i < c.V ? c.cur[i] : 0u;
  uint32_t total;
  const uint32_t o = c.vtile[blockIdx.x] + tile_excl_scan(d, s_warp, &total);
  if (i >= c.V) return;
  c.off[i] = o;
  c.cur[i] = o;
  if (i == c.V - 1) c.off[c.V] = o + d;
}

// short segments sorted in place by their own thread; longer ones listed for a CTA
__global__ void __launch_bounds__(kSmThreads) sm_csr_sort_kernel(SmCsr c, int32_t *err) {
  const uint32_t i = blockIdx.x * kSmThreads + threadIdx.x;
  if (i >= c.V || *err) return;
  const uint32_t b = c.off[i], n = c.off[i + 1] - b;
  if (n <= kSmSortThread) {
    uint32_t *s = c.ent + b;
    for (uint32_t k = 1; k < n; ++k) {
      const uint32_t x = s[k];
      uint32_t j = k;
      for (; j > 0 && s[j - 1] > x; --j) s[j] = s[j - 1];
      s[j] = x;
    }
    return;
  }
  const bool huge = n > kSmSortCta;
  const uint32_t k = atomicAdd(huge ? &c.hdr->n_huge : &c.hdr->n_long, 1u);
  if (k < (huge ? c.hcap : c.lcap)) c.lst[(huge ? c.lcap : 0u) + k] = i;
  else atomicOr(err, kSmErrBound);
}

__global__ void __launch_bounds__(kSmSortCtaThreads) sm_csr_sort_long_kernel(SmCsr c) {
  __shared__ uint32_t s[kSmSortCta];
  if (*c.err) return;
  const uint32_t nl = min(c.hdr->n_long, c.lcap);
  for (uint32_t k = blockIdx.x; k < nl; k += gridDim.x) {
    const uint32_t v = c.lst[k], b = c.off[v], n = min(c.off[v + 1] - b, kSmSortCta);
    uint32_t p = 2;
    while (p < n) p <<= 1;   // n <= kSmSortCta: at most 12 steps
    for (uint32_t r = threadIdx.x; r < p; r += blockDim.x) s[r] = r < n ? c.ent[b + r] : 0xFFFFFFFFu;
    __syncthreads();
    block_bitonic_sort(s, p);
    for (uint32_t r = threadIdx.x; r < n; r += blockDim.x) c.ent[b + r] = s[r];
    __syncthreads();
  }
}

// Ascending sort of n (any) keys in global memory by one CTA: the bitonic network in which every comparator puts the
// smaller key at the lower index (a "flip" step, then half-cleaners), positions >= n acting as +inf, so comparators
// that reach them are skipped and nothing needs padding.
__device__ void sm_cta_sort_global(uint32_t *s, uint32_t n) {
  uint32_t p = 1;
  while (p < n) p <<= 1;   // n < 2^28: at most 28 steps
  const uint32_t half = p >> 1;
  for (uint32_t k = 2; k <= p; k <<= 1) {
    for (uint32_t j = k >> 1; j > 0; j >>= 1) {
      const bool flip = j == (k >> 1);
      for (uint32_t t = threadIdx.x; t < half; t += blockDim.x) {
        const uint32_t a = ((t & ~(j - 1)) << 1) | (t & (j - 1));
        const uint32_t b = flip ? (a & ~(k - 1)) + (k - 1) - (t & (j - 1)) : a | j;
        if (b >= n) continue;
        const uint32_t x = s[a], y = s[b];
        if (x > y) { s[a] = y; s[b] = x; }
      }
      __syncthreads();
    }
  }
}

__global__ void __launch_bounds__(kSmSortCtaThreads) sm_csr_sort_huge_kernel(SmCsr c) {
  if (*c.err) return;
  const uint32_t nh = min(c.hdr->n_huge, c.hcap);
  for (uint32_t k = blockIdx.x; k < nh; k += gridDim.x) {
    const uint32_t v = c.lst[c.lcap + k], b = c.off[v];
    sm_cta_sort_global(c.ent + b, min(c.off[v + 1] - b, c.emax - b));
  }
}

static uint32_t sm_tiles(uint64_t n, uint32_t per) { return (uint32_t)((n + per - 1) / per); }

// The shared CSR build: count, scan, offsets, scatter, segment sort.  cur and hdr are zeroed by the caller.
template <class Source>
static cudaError_t sm_build_csr(const Source &src, const SmCsr &c, int32_t *err, cudaStream_t st) {
  const uint32_t vt = sm_tiles(c.V, kSmThreads), st_tiles = sm_tiles(src.n, kSmThreads);
  if (st_tiles) sm_csr_fill_kernel<false><<<st_tiles, kSmThreads, 0, st>>>(src, c, err);
  sm_csr_tile_kernel<<<vt, kSmThreads, 0, st>>>(c);
  tile_scan_kernel<<<1, kTileScanThreads, 0, st>>>(c.vtile, vt, &c.hdr->n_entries);
  sm_csr_offset_kernel<<<vt, kSmThreads, 0, st>>>(c);
  if (st_tiles) sm_csr_fill_kernel<true><<<st_tiles, kSmThreads, 0, st>>>(src, c, err);
  sm_csr_sort_kernel<<<vt, kSmThreads, 0, st>>>(c, err);
  sm_csr_sort_long_kernel<<<min(c.lcap, kSmLongCtas), kSmSortCtaThreads, 0, st>>>(c);
  sm_csr_sort_huge_kernel<<<min(c.hcap, kSmHugeCtas), kSmSortCtaThreads, 0, st>>>(c);
  return cudaGetLastError();
}

struct SmPassArgs {
  SmoothSrc src;
  const uint32_t *off, *ent;
  uint32_t V, fields;
  int laplacian;
  double lam;
  double *dst[3];     // float64 destination of every field (state, or the output normals)
  float *dst32[3];    // or, in the last pass, the float32 output of positions / colours
  const int32_t *err;
};

__global__ void __launch_bounds__(kSmThreads) sm_pass_kernel(SmPassArgs a) {
  const uint32_t i = blockIdx.x * kSmThreads + threadIdx.x;
  if (i >= a.V || *a.err) return;
  const uint32_t b = a.off[i];
  double out[3][3];
  smooth_vertex(a.src, i, a.ent + b, a.off[i + 1] - b, a.laplacian != 0, a.lam, a.fields, out);
#pragma unroll
  for (int f = 0; f < 3; ++f) {
    if (!((a.fields >> f) & 1u)) continue;
    const size_t o = 3 * (size_t)i;
    if (a.dst32[f]) {
      a.dst32[f][o] = (float)out[f][0]; a.dst32[f][o + 1] = (float)out[f][1]; a.dst32[f][o + 2] = (float)out[f][2];
    } else {
      a.dst[f][o] = out[f][0]; a.dst[f][o + 1] = out[f][1]; a.dst[f][o + 2] = out[f][2];
    }
  }
}

__global__ void __launch_bounds__(kSmThreads) sm_tri_normal_kernel(const float *xyz, const int32_t *tri, uint32_t T,
                                                                   double *tn, const int32_t *err) {
  const uint32_t t = blockIdx.x * kSmThreads + threadIdx.x;
  if (t >= T || *err) return;
  double n[3];
  smooth_tri_normal(xyz, __ldg(tri + 3 * (size_t)t), __ldg(tri + 3 * (size_t)t + 1), __ldg(tri + 3 * (size_t)t + 2), n);
  tn[3 * (size_t)t] = n[0]; tn[3 * (size_t)t + 1] = n[1]; tn[3 * (size_t)t + 2] = n[2];
}

__global__ void __launch_bounds__(kSmThreads) sm_vertex_normal_kernel(SmCsr c, const double *tn, double *out) {
  const uint32_t i = blockIdx.x * kSmThreads + threadIdx.x;
  if (i >= c.V || *c.err) return;
  const uint32_t b = c.off[i];
  double n[3];
  smooth_vertex_normal(c.ent + b, c.off[i + 1] - b, tn, n);
  out[3 * (size_t)i] = n[0]; out[3 * (size_t)i + 1] = n[1]; out[3 * (size_t)i + 2] = n[2];
}

__global__ void sm_empty_kernel(int32_t *err, uint32_t T) {
  if (threadIdx.x == 0 && blockIdx.x == 0) *err = T > 0 ? kSmErrTriangle : 0;   // no vertices: every id is bad
}

// ---------------------------------------------------------------------------------------------------------------
// scratch layout
// ---------------------------------------------------------------------------------------------------------------
struct SmLayout {
  size_t hdr, keys, vals, off, cur, vtile, ent, lst, tn, state, total;
  uint32_t cap, emax, lcap, hcap;
  bool ok;
};

// appends count elements of elem bytes at a 256-byte boundary; ok goes false instead of wrapping around
static size_t sm_region(size_t &off, unsigned long long count, size_t elem, bool &ok) {
  const size_t at = off;
  if (count > (SIZE_MAX / 2 - off) / elem) { ok = false; return at; }
  off = align_up(off + (size_t)count * elem, 256);
  return at;
}

// smoothing (adjacency = true): the edge table, the adjacency CSR (<= 6T entries: two per distinct edge) and the
// float64 state of two passes; normals: the incidence CSR (3T entries) and the triangle normals
static SmLayout sm_layout(uint32_t V, uint32_t T, bool adjacency) {
  SmLayout L{};
  L.ok = true;
  const unsigned long long c = 4ull * T;   // m3's table: at most 3T distinct edges, a load factor of at most 3/4
  L.cap = adjacency ? (uint32_t)(c < 1024ull ? 1024ull : c) : 0u;
  L.emax = (adjacency ? 6u : 3u) * T;      // T <= 2^25: below 2^28
  L.lcap = L.emax / (kSmSortThread + 1) + 1;
  L.hcap = L.emax / (kSmSortCta + 1) + 1;
  size_t off = 0;
  L.hdr = sm_region(off, 1, sizeof(SmHeader), L.ok);
  L.keys = sm_region(off, L.cap, 8, L.ok);
  L.vals = sm_region(off, L.cap, 4, L.ok);
  L.off = sm_region(off, (unsigned long long)V + 1, 4, L.ok);
  L.cur = sm_region(off, V, 4, L.ok);
  L.vtile = sm_region(off, (unsigned long long)sm_tiles(V, kSmThreads) + 1, 4, L.ok);
  L.ent = sm_region(off, L.emax, 4, L.ok);
  L.lst = sm_region(off, (unsigned long long)L.lcap + L.hcap, 4, L.ok);
  L.tn = sm_region(off, adjacency ? 0ull : 3ull * T, 8, L.ok);
  L.state = sm_region(off, adjacency ? 2ull * 3ull * 3ull * V : 0ull, 8, L.ok);   // 2 buffers x 3 fields x [V][3]
  L.total = off;
  return L;
}

static bool sm_sizes_ok(uint32_t V, uint32_t T) { return V <= kSmMaxVertices && T <= kSmMaxTriangles; }

static SmCsr sm_csr(uint8_t *base, const SmLayout &L, uint32_t V, const int32_t *err) {
  SmCsr c;
  c.V = V;
  c.emax = L.emax;
  c.off = (uint32_t *)(base + L.off);
  c.cur = (uint32_t *)(base + L.cur);
  c.vtile = (uint32_t *)(base + L.vtile);
  c.ent = (uint32_t *)(base + L.ent);
  c.lst = (uint32_t *)(base + L.lst);
  c.lcap = L.lcap;
  c.hcap = L.hcap;
  c.hdr = (SmHeader *)(base + L.hdr);
  c.err = err;
  return c;
}

// zeroes the error word, the header and the degrees
static cudaError_t sm_reset(uint8_t *base, const SmLayout &L, uint32_t V, int32_t *err, cudaStream_t st) {
  cudaError_t e = cudaMemsetAsync(err, 0, sizeof(int32_t), st);
  if (e == cudaSuccess) e = cudaMemsetAsync(base + L.hdr, 0, sizeof(SmHeader), st);
  if (e == cudaSuccess) e = cudaMemsetAsync(base + L.cur, 0, (size_t)V * 4, st);
  return e;
}

}  // namespace d2pc

using namespace d2pc;

extern "C" int d2pc_mesh_smooth_scratch_bytes(uint32_t vertices, uint32_t triangles, size_t *bytes) {
  if (!bytes) return D2PC_ERR_INVALID_ARGUMENT;
  if (!sm_sizes_ok(vertices, triangles)) return D2PC_ERR_UNSUPPORTED;
  const SmLayout L = sm_layout(vertices, triangles, true);
  if (!L.ok) return D2PC_ERR_UNSUPPORTED;
  *bytes = L.total;
  return D2PC_OK;
}

extern "C" int d2pc_mesh_smooth_enqueue(const float *d_vtx_xyz, const float *d_vtx_rgb, const double *d_vtx_normals,
                                        uint32_t vertices, const int32_t *d_tri, uint32_t triangles, int method,
                                        uint32_t iterations, double lambda_filter, double mu, uint32_t scope,
                                        void *d_scratch, size_t scratch_bytes, float *d_out_xyz, float *d_out_rgb,
                                        double *d_out_normals, int32_t *d_error, void *stream) {
  if (method != D2PC_SMOOTH_SIMPLE && method != D2PC_SMOOTH_LAPLACIAN && method != D2PC_SMOOTH_TAUBIN)
    return D2PC_ERR_INVALID_ARGUMENT;
  const uint32_t all = D2PC_SMOOTH_VERTEX | D2PC_SMOOTH_NORMAL | D2PC_SMOOTH_COLOR;
  if (scope == 0 || (scope & ~all) != 0) return D2PC_ERR_INVALID_ARGUMENT;
  if (!std::isfinite(lambda_filter) || !std::isfinite(mu)) return D2PC_ERR_INVALID_ARGUMENT;
  if (!d_scratch || !d_error) return D2PC_ERR_INVALID_ARGUMENT;
  if (vertices > 0 && (!d_vtx_xyz || !d_vtx_rgb || !d_out_xyz || !d_out_rgb)) return D2PC_ERR_INVALID_ARGUMENT;
  if (vertices > 0 && (d_vtx_normals != nullptr) != (d_out_normals != nullptr)) return D2PC_ERR_INVALID_ARGUMENT;
  if (triangles > 0 && !d_tri) return D2PC_ERR_INVALID_ARGUMENT;
  if (((uintptr_t)d_scratch & 255u) != 0) return D2PC_ERR_INVALID_ARGUMENT;
  if (!sm_sizes_ok(vertices, triangles)) return D2PC_ERR_UNSUPPORTED;
  const SmLayout L = sm_layout(vertices, triangles, true);
  if (!L.ok) return D2PC_ERR_UNSUPPORTED;
  if (scratch_bytes < L.total) return D2PC_ERR_WORKSPACE_TOO_SMALL;
  cudaStream_t st = (cudaStream_t)stream;
  if (vertices == 0) {
    sm_empty_kernel<<<1, 32, 0, st>>>(d_error, triangles);
    D2PC_CHECK_LAUNCH();
    return D2PC_OK;
  }
  // fields (0 position, 1 normal, 2 colour) filtered: bit f; normals only when the mesh has them
  const uint32_t fields = scope & (d_vtx_normals ? all : (uint32_t)(D2PC_SMOOTH_VERTEX | D2PC_SMOOTH_COLOR));
  uint8_t *base = (uint8_t *)d_scratch;
  cudaError_t e = sm_reset(base, L, vertices, d_error, st);
  // the fields outside the scope (all of them with 0 iterations) are copied
  const uint32_t passes = iterations * (method == D2PC_SMOOTH_TAUBIN ? 2u : 1u);
  const uint32_t live = passes > 0 ? fields : 0u;
  const size_t v3 = (size_t)vertices * 3;
  if (e == cudaSuccess && !(live & 1u))
    e = cudaMemcpyAsync(d_out_xyz, d_vtx_xyz, v3 * 4, cudaMemcpyDeviceToDevice, st);
  if (e == cudaSuccess && d_vtx_normals && !(live & 2u))
    e = cudaMemcpyAsync(d_out_normals, d_vtx_normals, v3 * 8, cudaMemcpyDeviceToDevice, st);
  if (e == cudaSuccess && !(live & 4u))
    e = cudaMemcpyAsync(d_out_rgb, d_vtx_rgb, v3 * 4, cudaMemcpyDeviceToDevice, st);
  if (e != cudaSuccess) return record_cuda_error(e);
  const uint32_t vt = sm_tiles(vertices, kSmThreads), ct = sm_tiles(vertices > triangles ? vertices : triangles,
                                                                        kSmThreads);
  sm_check_kernel<<<ct, kSmThreads, 0, st>>>(d_vtx_xyz, (fields & 4u) ? d_vtx_rgb : nullptr,
                                              (fields & 2u) ? d_vtx_normals : nullptr, vertices, d_tri, triangles,
                                              d_error);
  D2PC_CHECK_LAUNCH();
  if (live == 0) return D2PC_OK;
  unsigned long long *keys = (unsigned long long *)(base + L.keys);
  e = cudaMemsetAsync(keys, 0xFF, (size_t)L.cap * 8, st);
  if (e == cudaSuccess) e = cudaMemsetAsync(base + L.vals, 0xFF, (size_t)L.cap * 4, st);
  if (e != cudaSuccess) return record_cuda_error(e);
  if (triangles > 0) {
    sm_edge_kernel<<<sm_tiles(triangles, kSmThreads), kSmThreads, 0, st>>>(d_tri, triangles, keys,
                                                                             (uint32_t *)(base + L.vals), L.cap,
                                                                             d_error);
    D2PC_CHECK_LAUNCH();
  }
  const SmCsr c = sm_csr(base, L, vertices, d_error);
  e = sm_build_csr(SmEdgeSource{keys, L.cap}, c, d_error, st);
  if (e != cudaSuccess) return record_cuda_error(e);
  // state buffers: [buffer][field][V][3]
  double *state = (double *)(base + L.state);
  auto buf = [&](uint32_t b, int f) { return state + ((size_t)b * 3 + (size_t)f) * v3; };
  SmPassArgs a;
  a.off = c.off;
  a.ent = c.ent;
  a.V = vertices;
  a.fields = live;
  a.err = d_error;
  a.src.xyz = d_vtx_xyz;
  a.src.rgb = d_vtx_rgb;
  a.src.nrm = d_vtx_normals;
  for (uint32_t p = 0; p < passes; ++p) {
    const bool last = p + 1 == passes;
    a.laplacian = method != D2PC_SMOOTH_SIMPLE;
    a.lam = method == D2PC_SMOOTH_TAUBIN && (p & 1u) ? mu : lambda_filter;
    for (int f = 0; f < 3; ++f) {
      const bool on = (live >> f) & 1u;
      a.src.state[f] = on && p > 0 ? buf((p - 1) & 1u, f) : nullptr;   // unfiltered fields: always the input
      a.dst[f] = on ? (last ? (f == 1 ? d_out_normals : nullptr) : buf(p & 1u, f)) : nullptr;
      a.dst32[f] = on && last && f != 1 ? (f == 0 ? d_out_xyz : d_out_rgb) : nullptr;
    }
    sm_pass_kernel<<<vt, kSmThreads, 0, st>>>(a);
    D2PC_CHECK_LAUNCH();
  }
  return D2PC_OK;
}

extern "C" int d2pc_mesh_vertex_normals_scratch_bytes(uint32_t vertices, uint32_t triangles, size_t *bytes) {
  if (!bytes) return D2PC_ERR_INVALID_ARGUMENT;
  if (!sm_sizes_ok(vertices, triangles)) return D2PC_ERR_UNSUPPORTED;
  const SmLayout L = sm_layout(vertices, triangles, false);
  if (!L.ok) return D2PC_ERR_UNSUPPORTED;
  *bytes = L.total;
  return D2PC_OK;
}

extern "C" int d2pc_mesh_vertex_normals_enqueue(const float *d_vtx_xyz, uint32_t vertices, const int32_t *d_tri,
                                                uint32_t triangles, void *d_scratch, size_t scratch_bytes,
                                                double *d_out_normals, int32_t *d_error, void *stream) {
  if (!d_scratch || !d_error) return D2PC_ERR_INVALID_ARGUMENT;
  if (vertices > 0 && (!d_vtx_xyz || !d_out_normals)) return D2PC_ERR_INVALID_ARGUMENT;
  if (triangles > 0 && !d_tri) return D2PC_ERR_INVALID_ARGUMENT;
  if (((uintptr_t)d_scratch & 255u) != 0) return D2PC_ERR_INVALID_ARGUMENT;
  if (!sm_sizes_ok(vertices, triangles)) return D2PC_ERR_UNSUPPORTED;
  const SmLayout L = sm_layout(vertices, triangles, false);
  if (!L.ok) return D2PC_ERR_UNSUPPORTED;
  if (scratch_bytes < L.total) return D2PC_ERR_WORKSPACE_TOO_SMALL;
  cudaStream_t st = (cudaStream_t)stream;
  if (vertices == 0) {
    sm_empty_kernel<<<1, 32, 0, st>>>(d_error, triangles);
    D2PC_CHECK_LAUNCH();
    return D2PC_OK;
  }
  uint8_t *base = (uint8_t *)d_scratch;
  cudaError_t e = sm_reset(base, L, vertices, d_error, st);
  if (e != cudaSuccess) return record_cuda_error(e);
  sm_check_kernel<<<sm_tiles(vertices > triangles ? vertices : triangles, kSmThreads), kSmThreads, 0, st>>>(
      d_vtx_xyz, nullptr, nullptr, vertices, d_tri, triangles, d_error);
  D2PC_CHECK_LAUNCH();
  const SmCsr c = sm_csr(base, L, vertices, d_error);
  e = sm_build_csr(SmCornerSource{d_tri, 3u * triangles}, c, d_error, st);
  if (e != cudaSuccess) return record_cuda_error(e);
  double *tn = (double *)(base + L.tn);
  if (triangles > 0) {
    sm_tri_normal_kernel<<<sm_tiles(triangles, kSmThreads), kSmThreads, 0, st>>>(d_vtx_xyz, d_tri, triangles, tn,
                                                                                   d_error);
    D2PC_CHECK_LAUNCH();
  }
  sm_vertex_normal_kernel<<<sm_tiles(vertices, kSmThreads), kSmThreads, 0, st>>>(c, tn, d_out_normals);
  D2PC_CHECK_LAUNCH();
  return D2PC_OK;
}
