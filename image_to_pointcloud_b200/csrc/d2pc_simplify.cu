// d2pc_simplify.cu -- row m2: simplification of ONE triangle mesh by vertex clustering (Open3D's
// SimplifyVertexClustering, with average or Lindstrom quadric placement).  Our own spec, frozen in
// oracle/d2pc_simplify_oracle.py:
//   index      the ax-2 voxel rule on the vertices: vmin = bmin - vs/2, idx = floor((v - vmin) / vs), < 2^21 per axis
//   vertices   one per occupied cluster, ordered by its lowest member vertex id (which also gives its vertex row)
//   average    means of the members' positions and colours; normals: the members' sum, normalised
//   quadric    per triangle (float64, translated by bmin) w = area, n = unit normal, d = -n.q0: A += w n n^T and
//              b += w d n into the cluster of each corner; x = -A^-1 b when det A > 1e-4 trace(A)^3 and x lies in the
//              cluster's own cell, else the average
//   triangles  remapped, collapsed ones dropped, rotated to start at the smallest id, first of each form kept
// Launch sequence (every count stays on the device; nothing synchronises the host):
//   d2pc_rows_bounds_enqueue    vertex bounds -> bmin
//   simp_setup_kernel           origin, fixed-point scale of the positions, counters
//   simp_claim_kernel           per vertex: finiteness, cluster key, probe of an open-addressed table of keys; the
//                               lowest member claims the slot's representative with atomicMin (a warp's raster run
//                               of equal keys probes once); max |colour| and |normal| for their scales
//   simp_head_kernel / scan     representatives (slot's minimum == self) counted per tile, scanned: cluster ids
//   simp_assign_kernel          representative -> cluster id of its slot, vertex row and key of the cluster
//   simp_accum_kernel           per vertex: RED.64 of fixed-point position, colour and (hi, lo) normal sums
//   simp_tri_prep_kernel        per triangle: id check, cluster triple, canonical rotation; area partial sums
//   simp_tri_scale_kernel       (quadric) sum of the partial areas in a fixed order -> the quadric scales
//   simp_tri_insert_kernel      canonical triple into a table of triangle indices, first occurrence by atomicMin;
//                               (quadric) 9 fixed-point RED.64 per corner
//   simp_tri_flag_kernel / scan survivors per tile, scanned
//   simp_tri_write_kernel       survivors in input order
//   simp_finish_kernel          per cluster: means, 3x3 solve, normalisation
// No floating-point atomics: every sum is a 64-bit integer sum, so the result repeats bit for bit.
#include <cmath>

#include "d2pc_device.cuh"
#include "d2pc_scan.cuh"

namespace d2pc {

constexpr int kSimpThreads = 256;
constexpr int kSimpBits = 21;
constexpr uint32_t kSimpNone = 0xFFFFFFFFu;
constexpr unsigned long long kSimpNoKey = 0xFFFFFFFFFFFFFFFFull;
constexpr uint32_t kSimpMaxVertices = 1u << 24;
constexpr uint32_t kSimpMaxTriangles = 1u << 31;
constexpr uint32_t kSimpQuadric = D2PC_SIMPLIFY_QUADRIC, kSimpNormals = D2PC_SIMPLIFY_NORMALS;
constexpr double kSimpDetRel = 1e-4;
// error word bits
constexpr int32_t kSimpErrIndex = 1, kSimpErrTriangle = 2, kSimpErrNonFinite = 4;

struct __align__(256) SimpHeader {
  double vmin[3];     // cluster index origin: bmin - vs/2
  double origin[3];   // fixed-point origin of the positions and the quadrics: bmin
  double scale_p;     // fixed-point scale of the positions (power of two)
  double scale_a, scale_b;   // of the quadric A and b sums
  unsigned long long cmax_bits, nmax_bits;   // max |colour|, max |normal| as float64 bits (non-negative: ordered)
  uint32_t n_clusters, n_tri;
};

struct SimpArgs {
  const float *xyz, *rgb;
  const double *nrm;            // or nullptr
  const long long *row;
  const int32_t *tri;
  uint32_t V, T, vcap, tcap, vtiles, ttiles;
  double vs, inv_vs;
  SimpHeader *hdr;
  unsigned long long *vkey;     // [vcap] cluster key of every slot
  uint32_t *vrep;               // [vcap] lowest member of every slot
  uint32_t *slot_cid;           // [vcap] cluster id of every occupied slot
  uint32_t *vslot;              // [V] slot of every vertex (kSimpNone: not finite / out of range)
  uint32_t *vcid;               // [V] cluster of every vertex
  uint32_t *vtile;              // [vtiles + 1]
  unsigned long long *ckey;     // [V] key of every cluster
  uint32_t *cnt;                // [V] members of every cluster
  unsigned long long *acc;      // [V][kSimpAcc] position, colour, normal (hi, lo), quadric sums
  double *tarea;                // [ttiles] partial area sums
  uint32_t *canon;              // [T][3] canonical cluster triple (canon[0] = kSimpNone: dropped)
  uint32_t *tslot;              // [T]
  uint32_t *ttab;               // [tcap] lowest triangle index of every canonical form
  uint32_t *ttile;              // [ttiles + 1]
  int32_t *err;
  float *oxyz, *orgb;
  double *onrm;
  long long *orow;
  int32_t *otri;
  uint32_t *vcount, *tcount;
};
// accumulator words per cluster: 0..2 position, 3..5 colour, 6..11 normal (hi x y z, lo x y z), 12..20 quadric
constexpr int kSimpAcc = 21;

__device__ __forceinline__ unsigned long long simp_hash(unsigned long long k) {
  k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
  return k;
}
__device__ __forceinline__ uint32_t simp_slot(unsigned long long h, uint32_t cap) {
  return (uint32_t)(((h >> 32) * (unsigned long long)cap) >> 32);
}
__device__ __forceinline__ void red_add_s64(unsigned long long *p, double v) {
  atomicAdd(p, (unsigned long long)__double2ll_rn(v));
}
// 2^(k - ex) with x < 2^ex (x >= 0, finite): the largest power of two that keeps x * scale below 2^k
__device__ __forceinline__ double simp_scale(double x, int k) {
  int ex = 0;
  if (x > 0.0) frexp(x, &ex);
  return ldexp(1.0, k - ex);
}

__global__ void simp_setup_kernel(SimpArgs a, const float *bounds) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  SimpHeader *h = a.hdr;
  const double half = a.vs * 0.5;
  double ext = 0.0;
  for (int c = 0; c < 3; ++c) {
    const double bmin = (double)bounds[c];
    h->vmin[c] = bmin - half;
    h->origin[c] = bmin;
    const double e = (double)bounds[3 + c] - bmin;
    if (e > ext) ext = e;
  }
  // V < 2^24 terms of at most ext * scale < 2^38 each: |sum| < 2^62; each term is rounded by at most 2^-38 * ext
  h->scale_p = simp_scale(ext, 38);
  h->scale_a = h->scale_b = 0.0;
  h->cmax_bits = h->nmax_bits = 0ull;
  h->n_clusters = h->n_tri = 0;
  *a.err = 0;
}

// one vertex per lane; a run of lanes with equal keys (raster neighbours of a lattice mesh) probes once
__global__ void __launch_bounds__(kSimpThreads) simp_claim_kernel(SimpArgs a) {
  const uint32_t i = blockIdx.x * kSimpThreads + threadIdx.x;
  const int lane = threadIdx.x & 31;
  unsigned long long key = kSimpNoKey;
  double cm = 0.0, nm = 0.0;
  if (i < a.V) {
    const float x0 = __ldg(a.xyz + 3 * (size_t)i), x1 = __ldg(a.xyz + 3 * (size_t)i + 1), x2 = __ldg(a.xyz + 3 * (size_t)i + 2);
    const float c0 = __ldg(a.rgb + 3 * (size_t)i), c1 = __ldg(a.rgb + 3 * (size_t)i + 1), c2 = __ldg(a.rgb + 3 * (size_t)i + 2);
    bool fin = isfinite(x0) && isfinite(x1) && isfinite(x2) && isfinite(c0) && isfinite(c1) && isfinite(c2);
    cm = fmax(fmax(fabs((double)c0), fabs((double)c1)), fabs((double)c2));
    if (a.nrm) {
      const double n0 = __ldg(a.nrm + 3 * (size_t)i), n1 = __ldg(a.nrm + 3 * (size_t)i + 1), n2 = __ldg(a.nrm + 3 * (size_t)i + 2);
      fin = fin && isfinite(n0) && isfinite(n1) && isfinite(n2);
      nm = fmax(fmax(fabs(n0), fabs(n1)), fabs(n2));
    }
    if (!fin) {
      atomicOr(a.err, kSimpErrNonFinite);
      cm = nm = 0.0;
    } else {
      const double lim = (double)(1 << kSimpBits);
      const double o0 = (double)x0 - a.hdr->vmin[0], o1 = (double)x1 - a.hdr->vmin[1], o2 = (double)x2 - a.hdr->vmin[2];
      // floor((v - vmin) / vs) with the correctly rounded quotient (offsets >= 0), as in the ax-2 insert kernel
      const double i0 = floor(div_by_const_fast(o0, a.vs, a.inv_vs)), i1 = floor(div_by_const_fast(o1, a.vs, a.inv_vs)),
                   i2 = floor(div_by_const_fast(o2, a.vs, a.inv_vs));
      if (i0 >= 0.0 && i0 < lim && i1 >= 0.0 && i1 < lim && i2 >= 0.0 && i2 < lim)
        key = ((unsigned long long)i0 << (2 * kSimpBits)) | ((unsigned long long)i1 << kSimpBits) | (unsigned long long)i2;
      else
        atomicOr(a.err, kSimpErrIndex);   // "voxel_size is too small."
    }
  }
  // scales of the colour and normal sums: max as ordered float64 bits (no floating-point atomics)
  unsigned long long cb = (unsigned long long)__double_as_longlong(cm), nb = (unsigned long long)__double_as_longlong(nm);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    cb = max(cb, (unsigned long long)__shfl_xor_sync(0xffffffffu, cb, o));
    nb = max(nb, (unsigned long long)__shfl_xor_sync(0xffffffffu, nb, o));
  }
  if (lane == 0) {
    if (cb) atomicMax(&a.hdr->cmax_bits, cb);
    if (nb) atomicMax(&a.hdr->nmax_bits, nb);
  }
  const unsigned long long left = __shfl_up_sync(0xffffffffu, key, 1);
  const bool head = lane == 0 || left != key;
  const unsigned heads = __ballot_sync(0xffffffffu, head);
  uint32_t slot = kSimpNone;
  if (head && key != kSimpNoKey) {
    slot = simp_slot(simp_hash(key), a.vcap);
    while (true) {
      const unsigned long long prev = atomicCAS(a.vkey + slot, kSimpNoKey, key);
      if (prev == kSimpNoKey || prev == key) break;
      slot = slot + 1u == a.vcap ? 0u : slot + 1u;
    }
    atomicMin(a.vrep + slot, i);   // the run's first lane is its lowest vertex
  }
  const int start = 31 - __clz(heads & (0xffffffffu >> (31 - lane)));
  slot = __shfl_sync(0xffffffffu, slot, start);
  if (i < a.V) a.vslot[i] = key == kSimpNoKey ? kSimpNone : slot;
}

__device__ __forceinline__ bool simp_is_head(const SimpArgs &a, uint32_t i) {
  if (i >= a.V) return false;
  const uint32_t s = a.vslot[i];
  return s != kSimpNone && a.vrep[s] == i;
}

__global__ void __launch_bounds__(kSimpThreads) simp_head_kernel(SimpArgs a) {
  const uint32_t n = __syncthreads_count(simp_is_head(a, blockIdx.x * kSimpThreads + threadIdx.x));
  if (threadIdx.x == 0) a.vtile[blockIdx.x] = n;
}

__global__ void __launch_bounds__(kSimpThreads) simp_assign_kernel(SimpArgs a) {
  __shared__ uint32_t s_warp[kSimpThreads / 32];
  const uint32_t i = blockIdx.x * kSimpThreads + threadIdx.x;
  const bool head = simp_is_head(a, i);
  uint32_t total;
  const uint32_t id = a.vtile[blockIdx.x] + tile_excl_scan(head ? 1u : 0u, s_warp, &total);
  if (!head) return;
  const uint32_t s = a.vslot[i];
  a.slot_cid[s] = id;
  a.ckey[id] = a.vkey[s];
  a.orow[id] = a.row[i];
}

__global__ void __launch_bounds__(kSimpThreads) simp_accum_kernel(SimpArgs a) {
  const uint32_t i = blockIdx.x * kSimpThreads + threadIdx.x;
  if (i >= a.V) return;
  const uint32_t s = a.vslot[i];
  const uint32_t cid = s == kSimpNone ? kSimpNone : a.slot_cid[s];
  a.vcid[i] = cid;
  if (cid == kSimpNone) return;
  const SimpHeader *h = a.hdr;
  unsigned long long *acc = a.acc + (size_t)kSimpAcc * cid;
  atomicAdd(a.cnt + cid, 1u);
  const double sp = h->scale_p;
  // colours: V < 2^24 terms below 2^38 each; integral colours are exact (the scale is a power of two >= 1 for |c| < 2^38)
  const double sc = simp_scale(__longlong_as_double((long long)h->cmax_bits), 38);
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    red_add_s64(acc + k, ((double)__ldg(a.xyz + 3 * (size_t)i + k) - h->origin[k]) * sp);
    red_add_s64(acc + 3 + k, (double)__ldg(a.rgb + 3 * (size_t)i + k) * sc);
  }
  if (a.nrm) {
    // two words per component: hi = the nearest integer of n * sn (38 bits), lo = 38 more bits of what is left.
    // hi's remainder is exact (|r| <= 1/2), so each term is kept to 2^-77 * max|n| and the sums to far below 1e-9 rad
    const double sn = simp_scale(__longlong_as_double((long long)h->nmax_bits), 38);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const double x = __ldg(a.nrm + 3 * (size_t)i + k) * sn;
      const double hi = rint(x);
      atomicAdd(acc + 6 + k, (unsigned long long)(long long)hi);
      red_add_s64(acc + 9 + k, (x - hi) * 274877906944.0);   // 2^38
    }
  }
}

struct SimpD3 { double x, y, z; };

__device__ __forceinline__ SimpD3 simp_q(const SimpArgs &a, uint32_t v) {
  return {(double)__ldg(a.xyz + 3 * (size_t)v) - a.hdr->origin[0], (double)__ldg(a.xyz + 3 * (size_t)v + 1) - a.hdr->origin[1],
          (double)__ldg(a.xyz + 3 * (size_t)v + 2) - a.hdr->origin[2]};
}

// the triangle's plane in translated coordinates; false for a zero cross product
__device__ __forceinline__ bool simp_plane(const SimpArgs &a, const int32_t t[3], double *w, SimpD3 *n, double *d) {
  const SimpD3 q0 = simp_q(a, (uint32_t)t[0]), q1 = simp_q(a, (uint32_t)t[1]), q2 = simp_q(a, (uint32_t)t[2]);
  const SimpD3 e1{q1.x - q0.x, q1.y - q0.y, q1.z - q0.z}, e2{q2.x - q0.x, q2.y - q0.y, q2.z - q0.z};
  const SimpD3 c{e1.y * e2.z - e1.z * e2.y, e1.z * e2.x - e1.x * e2.z, e1.x * e2.y - e1.y * e2.x};
  const double cc = c.x * c.x + c.y * c.y + c.z * c.z;
  if (cc == 0.0) return false;
  const double ln = sqrt(cc);
  *w = ln * 0.5;
  *n = {c.x / ln, c.y / ln, c.z / ln};
  *d = -(n->x * q0.x + n->y * q0.y + n->z * q0.z);
  return true;
}

__device__ __forceinline__ bool simp_load_tri(const SimpArgs &a, uint32_t t, int32_t v[3]) {
#pragma unroll
  for (int k = 0; k < 3; ++k) v[k] = __ldg(a.tri + 3 * (size_t)t + k);
  return v[0] >= 0 && (uint32_t)v[0] < a.V && v[1] >= 0 && (uint32_t)v[1] < a.V && v[2] >= 0 && (uint32_t)v[2] < a.V;
}

template <bool QUADRIC>
__global__ void __launch_bounds__(kSimpThreads) simp_tri_prep_kernel(SimpArgs a) {
  __shared__ double s_area[kSimpThreads];
  const uint32_t t = blockIdx.x * kSimpThreads + threadIdx.x;
  double area = 0.0;
  if (t < a.T) {
    int32_t v[3];
    uint32_t c0 = kSimpNone, c1 = kSimpNone, c2 = kSimpNone;
    if (!simp_load_tri(a, t, v)) {
      atomicOr(a.err, kSimpErrTriangle);
    } else {
      c0 = a.vcid[v[0]]; c1 = a.vcid[v[1]]; c2 = a.vcid[v[2]];
      if (QUADRIC) {
        double w, d;
        SimpD3 n;
        if (c0 != kSimpNone && c1 != kSimpNone && c2 != kSimpNone && simp_plane(a, v, &w, &n, &d)) area = w;
      }
    }
    uint32_t *o = a.canon + 3 * (size_t)t;
    if (c0 == kSimpNone || c1 == kSimpNone || c2 == kSimpNone || c0 == c1 || c1 == c2 || c0 == c2) {
      o[0] = kSimpNone;
    } else if (c0 < c1 && c0 < c2) {
      o[0] = c0; o[1] = c1; o[2] = c2;
    } else if (c1 < c2) {
      o[0] = c1; o[1] = c2; o[2] = c0;
    } else {
      o[0] = c2; o[1] = c0; o[2] = c1;
    }
  }
  if (!QUADRIC) return;
  // fixed-order tree: the partial sums, and so the scales, repeat bit for bit
  s_area[threadIdx.x] = area;
  __syncthreads();
  for (int s = kSimpThreads / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) s_area[threadIdx.x] += s_area[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) a.tarea[blockIdx.x] = s_area[0];
}

__global__ void __launch_bounds__(kSimpThreads) simp_tri_scale_kernel(SimpArgs a) {
  __shared__ double s_sum[kSimpThreads];
  double s = 0.0;
  for (uint32_t k = threadIdx.x; k < a.ttiles; k += kSimpThreads) s += a.tarea[k];
  s_sum[threadIdx.x] = s;
  __syncthreads();
  for (int st = kSimpThreads / 2; st > 0; st >>= 1) {
    if (threadIdx.x < st) s_sum[threadIdx.x] += s_sum[threadIdx.x + st];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    // a cluster's |A_ij| sum is at most 3 * (total area) (each triangle adds once per corner), its |b_i| sum at most
    // that times max |d| <= sqrt(3) * extent <= sqrt(3) * 2^38 / scale_p; one part in 2^20 of slack covers the
    // rounding of the total: every sum stays below 2^61
    const double bound_a = 3.0 * s_sum[0] * (1.0 + 0x1p-20);
    a.hdr->scale_a = simp_scale(bound_a, 61);
    a.hdr->scale_b = simp_scale(bound_a * 1.7320508075688774 * ldexp(1.0, 38) / a.hdr->scale_p * (1.0 + 0x1p-20), 61);
  }
}

template <bool QUADRIC>
__global__ void __launch_bounds__(kSimpThreads) simp_tri_insert_kernel(SimpArgs a) {
  const uint32_t t = blockIdx.x * kSimpThreads + threadIdx.x;
  if (t >= a.T) return;
  const uint32_t *o = a.canon + 3 * (size_t)t;
  const uint32_t c0 = o[0];
  if (c0 != kSimpNone) {
    const uint32_t c1 = o[1], c2 = o[2];
    uint32_t slot = simp_slot(simp_hash(((unsigned long long)c0 << 32 | c1) ^ simp_hash(c2 + 0x9e3779b97f4a7c15ull)), a.tcap);
    while (true) {
      const uint32_t prev = atomicCAS(a.ttab + slot, kSimpNone, t);
      if (prev == kSimpNone) break;
      const uint32_t *p = a.canon + 3 * (size_t)prev;   // written by the previous launch
      if (p[0] == c0 && p[1] == c1 && p[2] == c2) { atomicMin(a.ttab + slot, t); break; }
      slot = slot + 1u == a.tcap ? 0u : slot + 1u;
    }
    a.tslot[t] = slot;
  }
  if (!QUADRIC) return;
  int32_t v[3];
  if (!simp_load_tri(a, t, v)) return;
  const uint32_t cc[3] = {a.vcid[v[0]], a.vcid[v[1]], a.vcid[v[2]]};
  if (cc[0] == kSimpNone || cc[1] == kSimpNone || cc[2] == kSimpNone) return;
  double w, d;
  SimpD3 n;
  if (!simp_plane(a, v, &w, &n, &d)) return;
  const double wn0 = w * n.x, wn1 = w * n.y, wn2 = w * n.z, wd = w * d;
  const double q[9] = {wn0 * n.x, wn0 * n.y, wn0 * n.z, wn1 * n.y, wn1 * n.z, wn2 * n.z, wd * n.x, wd * n.y, wd * n.z};
  const double sa = a.hdr->scale_a, sb = a.hdr->scale_b;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    unsigned long long *acc = a.acc + (size_t)kSimpAcc * cc[k] + 12;
#pragma unroll
    for (int j = 0; j < 9; ++j) red_add_s64(acc + j, q[j] * (j < 6 ? sa : sb));
  }
}

__device__ __forceinline__ bool simp_tri_kept(const SimpArgs &a, uint32_t t) {
  return t < a.T && a.canon[3 * (size_t)t] != kSimpNone && a.ttab[a.tslot[t]] == t;
}

__global__ void __launch_bounds__(kSimpThreads) simp_tri_flag_kernel(SimpArgs a) {
  const uint32_t n = __syncthreads_count(simp_tri_kept(a, blockIdx.x * kSimpThreads + threadIdx.x));
  if (threadIdx.x == 0) a.ttile[blockIdx.x] = n;
}

__global__ void __launch_bounds__(kSimpThreads) simp_tri_write_kernel(SimpArgs a) {
  __shared__ uint32_t s_warp[kSimpThreads / 32];
  const uint32_t t = blockIdx.x * kSimpThreads + threadIdx.x;
  const bool keep = simp_tri_kept(a, t);
  uint32_t total;
  const uint32_t j = a.ttile[blockIdx.x] + tile_excl_scan(keep ? 1u : 0u, s_warp, &total);
  if (!keep) return;
#pragma unroll
  for (int k = 0; k < 3; ++k) a.otri[3 * (size_t)j + k] = (int32_t)a.canon[3 * (size_t)t + k];
}

__device__ __forceinline__ double simp_word(const unsigned long long *acc, int k) { return (double)(long long)acc[k]; }

template <bool QUADRIC, bool NORMALS>
__global__ void __launch_bounds__(kSimpThreads) simp_finish_kernel(SimpArgs a) {
  const uint32_t c = blockIdx.x * kSimpThreads + threadIdx.x;
  if (c >= a.hdr->n_clusters) return;
  const SimpHeader *h = a.hdr;
  const unsigned long long *acc = a.acc + (size_t)kSimpAcc * c;
  const double n = (double)a.cnt[c];
  const double inv_p = 1.0 / h->scale_p;   // powers of two: exact
  const double inv_c = 1.0 / simp_scale(__longlong_as_double((long long)h->cmax_bits), 38);
  double x[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    // the sums are exact multiples of the quanta and convert exactly (< 2^53 quanta for integral colours): the colour
    // means of integral colours are the correctly rounded exact means
    x[k] = h->origin[k] + simp_word(acc, k) * inv_p / n;
    a.orgb[3 * (size_t)c + k] = (float)(simp_word(acc, 3 + k) * inv_c / n);
  }
  if (QUADRIC) {
    const double ia = 1.0 / h->scale_a, ib = 1.0 / h->scale_b;
    const double a00 = simp_word(acc, 12) * ia, a01 = simp_word(acc, 13) * ia, a02 = simp_word(acc, 14) * ia,
                 a11 = simp_word(acc, 15) * ia, a12 = simp_word(acc, 16) * ia, a22 = simp_word(acc, 17) * ia;
    const double b0 = simp_word(acc, 18) * ib, b1 = simp_word(acc, 19) * ib, b2 = simp_word(acc, 20) * ib;
    const double c00 = a11 * a22 - a12 * a12, c01 = a02 * a12 - a01 * a22, c02 = a01 * a12 - a02 * a11;
    const double c11 = a00 * a22 - a02 * a02, c12 = a01 * a02 - a00 * a12, c22 = a00 * a11 - a01 * a01;
    const double det = (a00 * c00 + a01 * c01) + a02 * c02;
    const double tr = (a00 + a11) + a22;
    if (tr > 0.0 && det > kSimpDetRel * tr * tr * tr) {
      const double q[3] = {-((c00 * b0 + c01 * b1) + c02 * b2) / det + h->origin[0],
                           -((c01 * b0 + c11 * b1) + c12 * b2) / det + h->origin[1],
                           -((c02 * b0 + c12 * b1) + c22 * b2) / det + h->origin[2]};
      const unsigned long long key = a.ckey[c];
      const double idx[3] = {(double)(key >> (2 * kSimpBits)), (double)((key >> kSimpBits) & ((1u << kSimpBits) - 1u)),
                             (double)(key & ((1u << kSimpBits) - 1u))};
      bool inside = true;
#pragma unroll
      for (int k = 0; k < 3; ++k)
        inside = inside && q[k] >= h->vmin[k] + idx[k] * a.vs && q[k] <= h->vmin[k] + (idx[k] + 1.0) * a.vs;
      if (inside) { x[0] = q[0]; x[1] = q[1]; x[2] = q[2]; }
    }
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) a.oxyz[3 * (size_t)c + k] = (float)x[k];
  if (NORMALS) {
    const double inv_n = 1.0 / simp_scale(__longlong_as_double((long long)h->nmax_bits), 38);
    double s[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) s[k] = simp_word(acc, 6 + k) * inv_n + simp_word(acc, 9 + k) * (inv_n * 0x1p-38);
    const double nn = s[0] * s[0] + s[1] * s[1] + s[2] * s[2];
    const double ln = sqrt(nn);
#pragma unroll
    for (int k = 0; k < 3; ++k) a.onrm[3 * (size_t)c + k] = nn == 0.0 ? 0.0 : s[k] / ln;
  }
}

// publishes the counts; an error leaves none
__global__ void simp_done_kernel(SimpArgs a) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const bool bad = *a.err != 0;
  *a.vcount = bad ? 0u : a.hdr->n_clusters;
  *a.tcount = bad ? 0u : a.hdr->n_tri;
}

__global__ void simp_count_kernel(uint32_t *count, uint32_t n) {
  if (threadIdx.x == 0 && blockIdx.x == 0) *count = n;
}

__global__ void simp_empty_kernel(int32_t *err, uint32_t T, uint32_t *vcount, uint32_t *tcount) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  *err = T > 0 ? kSimpErrTriangle : 0;   // with no vertices every triangle id is out of range
  *vcount = 0;
  *tcount = 0;
}

struct SimpLayout {
  size_t hdr, vkey, vrep, slot_cid, vslot, vcid, vtile, ckey, cnt, acc, tarea, canon, tslot, ttab, ttile, bounds, total;
  uint32_t vcap, tcap, vtiles, ttiles;
};

static uint32_t simp_cap(uint32_t n) {
  const unsigned long long c = 2ull * n;
  return (uint32_t)(c < 1024ull ? 1024ull : c);
}

static SimpLayout simp_layout(uint32_t V, uint32_t T) {
  SimpLayout L;
  L.vcap = simp_cap(V);
  L.tcap = simp_cap(T);
  L.vtiles = (V + kSimpThreads - 1) / kSimpThreads;
  L.ttiles = (uint32_t)(((unsigned long long)T + kSimpThreads - 1) / kSimpThreads);
  size_t off = 0;
  L.hdr = off;      off = align_up(off + sizeof(SimpHeader), 256);
  L.bounds = off;   off = align_up(off + 6 * sizeof(float) + 7 * sizeof(uint32_t), 256);
  L.vkey = off;     off = align_up(off + (size_t)L.vcap * 8, 256);
  L.vrep = off;     off = align_up(off + (size_t)L.vcap * 4, 256);
  L.slot_cid = off; off = align_up(off + (size_t)L.vcap * 4, 256);
  L.vslot = off;    off = align_up(off + (size_t)V * 4, 256);
  L.vcid = off;     off = align_up(off + (size_t)V * 4, 256);
  L.vtile = off;    off = align_up(off + ((size_t)L.vtiles + 1) * 4, 256);
  L.ckey = off;     off = align_up(off + (size_t)V * 8, 256);
  L.cnt = off;      off = align_up(off + (size_t)V * 4, 256);
  L.acc = off;      off = align_up(off + (size_t)V * kSimpAcc * 8, 256);
  L.tarea = off;    off = align_up(off + ((size_t)L.ttiles + 1) * 8, 256);
  L.canon = off;    off = align_up(off + (size_t)T * 12, 256);
  L.tslot = off;    off = align_up(off + (size_t)T * 4, 256);
  L.ttab = off;     off = align_up(off + (size_t)L.tcap * 4, 256);
  L.ttile = off;    off = align_up(off + ((size_t)L.ttiles + 1) * 4, 256);
  L.total = off;
  return L;
}

static bool simp_sizes_ok(uint32_t V, uint32_t T) { return V < kSimpMaxVertices && T < kSimpMaxTriangles; }

}  // namespace d2pc

using namespace d2pc;

extern "C" int d2pc_mesh_simplify_scratch_bytes(uint32_t vertices, uint32_t triangles, size_t *bytes) {
  if (!bytes) return D2PC_ERR_INVALID_ARGUMENT;
  if (!simp_sizes_ok(vertices, triangles)) return D2PC_ERR_UNSUPPORTED;
  *bytes = simp_layout(vertices, triangles).total;
  return D2PC_OK;
}

extern "C" int d2pc_mesh_simplify_enqueue(const float *d_vtx_xyz, const float *d_vtx_rgb, const double *d_vtx_normals,
                                          const int64_t *d_vtx_row, uint32_t vertices, const int32_t *d_tri,
                                          uint32_t triangles, double voxel_size, uint32_t flags, void *d_scratch,
                                          size_t scratch_bytes, float *d_out_xyz, float *d_out_rgb,
                                          double *d_out_normals, int64_t *d_out_row, uint32_t *d_out_vtx_count,
                                          int32_t *d_out_tri, uint32_t *d_out_tri_count, int32_t *d_error,
                                          void *stream) {
  if (!(std::isfinite(voxel_size) && voxel_size > 0.0)) return D2PC_ERR_INVALID_ARGUMENT;
  if ((flags & ~(kSimpQuadric | kSimpNormals)) != 0) return D2PC_ERR_INVALID_ARGUMENT;
  if (!d_scratch || !d_out_vtx_count || !d_out_tri_count || !d_error) return D2PC_ERR_INVALID_ARGUMENT;
  if (vertices > 0 && (!d_vtx_xyz || !d_vtx_rgb || !d_vtx_row || !d_out_xyz || !d_out_rgb || !d_out_row))
    return D2PC_ERR_INVALID_ARGUMENT;
  if ((flags & kSimpNormals) && vertices > 0 && (!d_vtx_normals || !d_out_normals)) return D2PC_ERR_INVALID_ARGUMENT;
  if (triangles > 0 && (!d_tri || !d_out_tri)) return D2PC_ERR_INVALID_ARGUMENT;
  if (((uintptr_t)d_scratch & 255u) != 0) return D2PC_ERR_INVALID_ARGUMENT;
  if (!simp_sizes_ok(vertices, triangles)) return D2PC_ERR_UNSUPPORTED;
  const SimpLayout L = simp_layout(vertices, triangles);
  if (scratch_bytes < L.total) return D2PC_ERR_WORKSPACE_TOO_SMALL;
  cudaStream_t st = (cudaStream_t)stream;
  if (vertices == 0) {
    simp_empty_kernel<<<1, 32, 0, st>>>(d_error, triangles, d_out_vtx_count, d_out_tri_count);
    D2PC_CHECK_LAUNCH();
    return D2PC_OK;
  }
  uint8_t *base = (uint8_t *)d_scratch;
  const bool quadric = (flags & kSimpQuadric) != 0, normals = (flags & kSimpNormals) != 0;
  SimpArgs a;
  a.xyz = d_vtx_xyz;
  a.rgb = d_vtx_rgb;
  a.nrm = normals ? d_vtx_normals : nullptr;
  a.row = (const long long *)d_vtx_row;
  a.tri = d_tri;
  a.V = vertices;
  a.T = triangles;
  a.vcap = L.vcap;
  a.tcap = L.tcap;
  a.vtiles = L.vtiles;
  a.ttiles = L.ttiles;
  a.vs = voxel_size;
  a.inv_vs = 1.0 / voxel_size;
  a.hdr = (SimpHeader *)(base + L.hdr);
  a.vkey = (unsigned long long *)(base + L.vkey);
  a.vrep = (uint32_t *)(base + L.vrep);
  a.slot_cid = (uint32_t *)(base + L.slot_cid);
  a.vslot = (uint32_t *)(base + L.vslot);
  a.vcid = (uint32_t *)(base + L.vcid);
  a.vtile = (uint32_t *)(base + L.vtile);
  a.ckey = (unsigned long long *)(base + L.ckey);
  a.cnt = (uint32_t *)(base + L.cnt);
  a.acc = (unsigned long long *)(base + L.acc);
  a.tarea = (double *)(base + L.tarea);
  a.canon = (uint32_t *)(base + L.canon);
  a.tslot = (uint32_t *)(base + L.tslot);
  a.ttab = (uint32_t *)(base + L.ttab);
  a.ttile = (uint32_t *)(base + L.ttile);
  a.err = d_error;
  a.oxyz = d_out_xyz;
  a.orgb = d_out_rgb;
  a.onrm = d_out_normals;
  a.orow = (long long *)d_out_row;
  a.otri = d_out_tri;
  a.vcount = d_out_vtx_count;
  a.tcount = d_out_tri_count;
  float *bounds = (float *)(base + L.bounds);
  uint32_t *bkeys = (uint32_t *)(bounds + 6);
  uint32_t *bcount = bkeys + 6;   // the bounds kernel reads its row count from the device
  simp_count_kernel<<<1, 32, 0, st>>>(bcount, vertices);
  D2PC_CHECK_LAUNCH();
  const int rc = d2pc_rows_bounds_enqueue(d_vtx_xyz, bcount, vertices, bkeys, bounds, stream);
  if (rc) return rc;
  cudaError_t e = cudaMemsetAsync(a.vkey, 0xFF, (size_t)L.vcap * 8, st);
  if (e == cudaSuccess) e = cudaMemsetAsync(a.vrep, 0xFF, (size_t)L.vcap * 4, st);
  if (e == cudaSuccess) e = cudaMemsetAsync(a.cnt, 0, (size_t)vertices * 4, st);
  if (e == cudaSuccess) e = cudaMemsetAsync(a.acc, 0, (size_t)vertices * kSimpAcc * 8, st);
  if (e == cudaSuccess && triangles > 0) e = cudaMemsetAsync(a.ttab, 0xFF, (size_t)L.tcap * 4, st);
  if (e != cudaSuccess) return record_cuda_error(e);
  simp_setup_kernel<<<1, 32, 0, st>>>(a, bounds);
  D2PC_CHECK_LAUNCH();
  simp_claim_kernel<<<L.vtiles, kSimpThreads, 0, st>>>(a);
  D2PC_CHECK_LAUNCH();
  simp_head_kernel<<<L.vtiles, kSimpThreads, 0, st>>>(a);
  D2PC_CHECK_LAUNCH();
  tile_scan_kernel<<<1, kTileScanThreads, 0, st>>>(a.vtile, L.vtiles, &a.hdr->n_clusters);
  D2PC_CHECK_LAUNCH();
  simp_assign_kernel<<<L.vtiles, kSimpThreads, 0, st>>>(a);
  D2PC_CHECK_LAUNCH();
  simp_accum_kernel<<<L.vtiles, kSimpThreads, 0, st>>>(a);
  D2PC_CHECK_LAUNCH();
  if (triangles > 0) {
    if (quadric) simp_tri_prep_kernel<true><<<L.ttiles, kSimpThreads, 0, st>>>(a);
    else simp_tri_prep_kernel<false><<<L.ttiles, kSimpThreads, 0, st>>>(a);
    D2PC_CHECK_LAUNCH();
    if (quadric) {
      simp_tri_scale_kernel<<<1, kSimpThreads, 0, st>>>(a);
      D2PC_CHECK_LAUNCH();
      simp_tri_insert_kernel<true><<<L.ttiles, kSimpThreads, 0, st>>>(a);
    } else {
      simp_tri_insert_kernel<false><<<L.ttiles, kSimpThreads, 0, st>>>(a);
    }
    D2PC_CHECK_LAUNCH();
    simp_tri_flag_kernel<<<L.ttiles, kSimpThreads, 0, st>>>(a);
    D2PC_CHECK_LAUNCH();
    tile_scan_kernel<<<1, kTileScanThreads, 0, st>>>(a.ttile, L.ttiles, &a.hdr->n_tri);
    D2PC_CHECK_LAUNCH();
    simp_tri_write_kernel<<<L.ttiles, kSimpThreads, 0, st>>>(a);
    D2PC_CHECK_LAUNCH();
  }
  if (quadric && triangles > 0) {
    if (normals) simp_finish_kernel<true, true><<<L.vtiles, kSimpThreads, 0, st>>>(a);
    else simp_finish_kernel<true, false><<<L.vtiles, kSimpThreads, 0, st>>>(a);
  } else {
    if (normals) simp_finish_kernel<false, true><<<L.vtiles, kSimpThreads, 0, st>>>(a);
    else simp_finish_kernel<false, false><<<L.vtiles, kSimpThreads, 0, st>>>(a);
  }
  D2PC_CHECK_LAUNCH();
  simp_done_kernel<<<1, 32, 0, st>>>(a);
  D2PC_CHECK_LAUNCH();
  return D2PC_OK;
}
