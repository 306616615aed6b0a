// d2pc_sor.cu -- row f1: statistical outlier removal, the step the reference runs right after the
// hot path (refine_point_cloud, backend/app.py:252-269 -> Open3D remove_statistical_outlier(
// nb_neighbors=20, std_ratio=2.0)).  Spec (Open3D geometry/PointCloud.cpp, restated in
// oracle/d2pc_oracle.py::statistical_outlier_removal; Open3D itself is not installed: parity unpinned):
//   avg[i]  = mean of sqrt(d2) over the k nearest points of i INCLUDING i itself, d2 accumulated
//             axis by axis in float64, summed in ascending order
//   mean    = sum(avg[avg > 0]) / N ;  std = sqrt(sum((avg - mean)^2 [avg > 0]) / (N - 1))
//   keep i  iff 0 < avg[i] < mean + std_ratio * std          (rows keep their order)
//
// Exact k-NN on the device with a HASHED uniform grid (only occupied cells exist):
//   begin    kSorTrials candidate cell sizes around (volume / n)^(1/3)
//   trial    for every candidate: insert the cell keys into the hash table, count the occupied cells;
//   choose   the finest cell size that still holds >= kSorTargetOcc points per occupied cell on average
//            (a surface fills far fewer cells than its bounding box has, a volume fills them all; the
//            occupancy, not the box, decides)
//   build    insert again with the chosen size: slot of every point, per-slot counts
//   scan     exclusive prefix over the table slots (block scan, scan of block sums, add)
//   scatter  points copied into slot order (float32 x, y, z) with their source rows
//   query    one thread per point IN SLOT ORDER (the lanes of a warp share candidate lists): own cell, then
//            shells of growing Chebyshev radius R, each neighbour cell found by one hash probe; a float32
//            estimate rejects most candidates before the exact float64 distance; the sorted list of the
//            k smallest d2 lives in local memory; the search stops as soon as the k-th distance is no
//            larger than the distance to everything unvisited, which makes the result exact
//   stats    deterministic two-pass reduction -> threshold
//   compact  per-tile kept counts, scan, ordered copy of kept rows + their source indices
#include <stdlib.h>
#include "d2pc_grid.cuh"

namespace d2pc {

__global__ void sor_begin_kernel(SorWs w, const uint32_t *count, const float *bounds) {
  if (threadIdx.x != 0) return;
  SorHeader *h = w.hdr;
  const uint32_t n = *count;
  h->n = n;
  double mx = 0.0, vol = 1.0;
  int nd = 0;
  for (int a = 0; a < 3; ++a) {
    const double lo = (double)bounds[a], hi = (double)bounds[3 + a];
    h->mn[a] = (n > 0 && lo == lo) ? lo : 0.0;
    h->ext[a] = (n > 0 && hi == hi && lo == lo && hi > lo) ? hi - lo : 0.0;
    if (h->ext[a] > mx) mx = h->ext[a];
    if (h->ext[a] > 0.0) { vol *= h->ext[a]; ++nd; }
  }
  // middle candidate: the size at which the non-degenerate box has about n cells; never finer than the
  // coordinate range allows
  double base = (n > 0 && nd > 0) ? pow(vol / (double)n, 1.0 / (double)nd) : 1.0;
  const double floor_h = mx > 0.0 ? mx / (double)((1 << kSorCoordBits) - 2) : 1.0;
  for (int t = 0; t < kSorTrials; ++t) {
    double ht = base * pow(kSorTrialStep, (double)(3 - t));  // t = 0 coarsest ... kSorTrials - 1 finest
    h->trial_h[t] = ht > floor_h ? ht : floor_h;
    h->trial_occ[t] = 0;
  }
  h->slack = 1e-9 * mx + 1e-300;
  h->n_heavy = 0;
  h->heavy_total = 0;
}

// Grid of one cell size given by the caller (density clustering, d2pc_cluster.cu).  Sets *err to
// D2PC_CLUSTER_ERR_GRID when an axis would need kSorCellLimit cells or more: sor_cell_coords clamps beyond that,
// and a clamped cell would merge points that are far apart.
__global__ void sor_fixed_begin_kernel(SorWs w, const uint32_t *count, const float *bounds, double cs, uint32_t *err) {
  if (threadIdx.x != 0) return;
  SorHeader *h = w.hdr;
  const uint32_t n = *count;
  h->n = n;
  double mx = 0.0;
  bool fits = true;
  for (int a = 0; a < 3; ++a) {
    const double lo = (double)bounds[a], hi = (double)bounds[3 + a];
    h->mn[a] = (n > 0 && lo == lo) ? lo : 0.0;
    h->ext[a] = (n > 0 && hi == hi && lo == lo && hi > lo) ? hi - lo : 0.0;
    if (h->ext[a] > mx) mx = h->ext[a];
    const double q = h->ext[a] / cs;
    fits = fits && q < kSorCellLimit;
    h->dim[a] = q < kSorCellLimit ? (int32_t)floor(q) + 1 : (int32_t)kSorCellLimit;
  }
  h->h = cs;
  h->chosen = 0;
  h->slack = 1e-9 * mx + 1e-300;
  h->n_heavy = 0;
  h->heavy_total = 0;
  *err = fits ? 0u : (uint32_t)D2PC_CLUSTER_ERR_GRID;
}

__global__ void sor_clear_kernel(SorWs w) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < w.cap; i += (size_t)gridDim.x * blockDim.x) {
    w.keys[i] = kSorEmpty;
    w.cell_cnt[i] = 0u;
  }
}

// occupied cells for candidate size `trial`
__global__ void __launch_bounds__(kSorThreads) sor_trial_kernel(SorWs w, const float *xyz, int trial) {
  __shared__ uint32_t s_new;
  if (threadIdx.x == 0) s_new = 0;
  __syncthreads();
  SorHeader *h = w.hdr;
  const uint32_t n = h->n;
  const double cs = h->trial_h[trial];
  uint32_t mine = 0;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    int32_t c[3];
    sor_cell_coords(h, cs, (double)__ldg(xyz + 3 * (size_t)i), (double)__ldg(xyz + 3 * (size_t)i + 1),
                    (double)__ldg(xyz + 3 * (size_t)i + 2), c);
    bool fresh;
    sor_insert(w, sor_key(c[0], c[1], c[2]), &fresh);
    mine += fresh ? 1u : 0u;
  }
  mine = warp_sum(mine);
  if ((threadIdx.x & 31) == 0 && mine) atomicAdd(&s_new, mine);
  __syncthreads();
  if (threadIdx.x == 0 && s_new) atomicAdd(&h->trial_occ[trial], s_new);
}

__global__ void sor_choose_kernel(SorWs w, double target_occ) {
  if (threadIdx.x != 0) return;
  SorHeader *h = w.hdr;
  int best = 0;
  for (int t = 0; t < kSorTrials; ++t) {
    const double occ = h->trial_occ[t] ? (double)h->n / (double)h->trial_occ[t] : 0.0;
    if (occ >= target_occ) best = t;  // finest size that still fills its cells
  }
  h->chosen = (uint32_t)best;
  h->h = h->trial_h[best];
  for (int a = 0; a < 3; ++a) {
    const double q = floor(h->ext[a] / h->h) + 1.0;
    h->dim[a] = q < 1048575.0 ? (int32_t)q : 1048575;
  }
}

__global__ void __launch_bounds__(kSorThreads) sor_count_kernel(SorWs w, const float *xyz) {
  const SorHeader *h = w.hdr;
  const uint32_t n = h->n;
  const double cs = h->h;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    int32_t c[3];
    sor_cell_coords(h, cs, (double)__ldg(xyz + 3 * (size_t)i), (double)__ldg(xyz + 3 * (size_t)i + 1),
                    (double)__ldg(xyz + 3 * (size_t)i + 2), c);
    bool fresh;
    const uint32_t slot = sor_insert(w, sor_key(c[0], c[1], c[2]), &fresh);
    w.pt_cell[i] = slot;
    atomicAdd(&w.cell_cnt[slot], 1u);
  }
}

// block-wide exclusive scan of one value per thread; returns the exclusive prefix, *total = block sum
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t *s_warp, uint32_t *total) {
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

// phase 1: per block of 1024 cells, exclusive prefix inside the block -> cell_off, block total -> blk_sum;
// the counts are zeroed so that the array can serve as the scatter cursors
__global__ void __launch_bounds__(kSorScanThreads) sor_scan1_kernel(SorWs w) {
  __shared__ uint32_t s_warp[32];
  const uint32_t nc = w.cap;
  const uint32_t i = blockIdx.x * (uint32_t)kSorScanThreads + threadIdx.x;
  if (blockIdx.x * (uint32_t)kSorScanThreads >= nc) return;
  const uint32_t v = i < nc ? w.cell_cnt[i] : 0u;
  uint32_t total;
  const uint32_t ex = block_excl_scan(v, s_warp, &total);
  if (i < nc) { w.cell_off[i] = ex; w.cell_cnt[i] = 0u; }
  if (threadIdx.x == 0) w.blk_sum[blockIdx.x] = total;
}
// phase 2: exclusive scan of the block sums by one CTA
__global__ void __launch_bounds__(kSorScanThreads) sor_scan2_kernel(SorWs w) {
  __shared__ uint32_t s_warp[32];
  __shared__ uint32_t s_carry;
  const uint32_t nb = (w.cap + kSorScanThreads - 1) / kSorScanThreads;
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  for (uint32_t base = 0; base < nb; base += kSorScanThreads) {
    const uint32_t i = base + threadIdx.x;
    const uint32_t v = i < nb ? w.blk_sum[i] : 0u;
    uint32_t total;
    const uint32_t ex = block_excl_scan(v, s_warp, &total);
    if (i < nb) w.blk_sum[i] = s_carry + ex;
    __syncthreads();
    if (threadIdx.x == 0) s_carry += total;
    __syncthreads();
  }
}
// phase 3: add the block offsets; the entry past the last cell holds n
__global__ void __launch_bounds__(kSorScanThreads) sor_scan3_kernel(SorWs w) {
  const uint32_t nc = w.cap;
  const uint32_t i = blockIdx.x * (uint32_t)kSorScanThreads + threadIdx.x;
  if (i < nc) w.cell_off[i] += w.blk_sum[blockIdx.x];
  if (i == nc) w.cell_off[nc] = w.hdr->n;
}

__global__ void __launch_bounds__(kSorThreads) sor_scatter_kernel(SorWs w, const float *xyz) {
  const uint32_t n = w.hdr->n;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint32_t cell = w.pt_cell[i];
    const uint32_t pos = w.cell_off[cell] + atomicAdd(&w.cell_cnt[cell], 1u);
#pragma unroll
    for (int k = 0; k < 3; ++k) w.sorted[3 * (size_t)pos + k] = __ldg(xyz + 3 * (size_t)i + k);
    w.sorted_idx[pos] = i;
  }
}

// ---- very heavy cells: list, offsets, per-cell sort by x ---------------------------------------------
__global__ void __launch_bounds__(256) sor_heavy_list_kernel(SorWs w) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < w.cap; i += (size_t)gridDim.x * blockDim.x) {
    const uint32_t c = w.cell_off[i + 1] - w.cell_off[i];
    w.cell_cnt[i] = 0u;   // free after the scatter: from here on it only carries the "sorted" flag
    if (c > kSorHeavyMin && c <= kSorHeavyMax) {
      const uint32_t k = atomicAdd(&w.hdr->n_heavy, 1u);
      if (k < kSorMaxHeavy) w.heavy[2 * k] = (uint32_t)i;
    }
  }
}
__device__ __forceinline__ uint32_t sor_pow2(uint32_t x) {
  uint32_t p = 1;
  while (p < x) p <<= 1;
  return p;
}
__global__ void sor_heavy_offsets_kernel(SorWs w) {
  if (threadIdx.x != 0) return;
  SorHeader *h = w.hdr;
  if (h->n_heavy > kSorMaxHeavy) h->n_heavy = kSorMaxHeavy;
  uint32_t off = 0;
  for (uint32_t k = 0; k < h->n_heavy; ++k) {
    const uint32_t slot = w.heavy[2 * k];
    w.heavy[2 * k + 1] = off;
    off += sor_pow2(w.cell_off[slot + 1] - w.cell_off[slot]);  // sum <= 2 n
  }
  h->heavy_total = off;
}
// one CTA per heavy cell: bitonic sort of (x key, rank) pairs in global memory (L2 resident), then the
// cell's segment of `sorted` / `sorted_idx` is permuted into x order and the cell is flagged as sorted
__global__ void __launch_bounds__(1024) sor_heavy_sort_kernel(SorWs w) {
  const uint32_t b = blockIdx.x;
  if (b >= w.hdr->n_heavy) return;
  const uint32_t slot = w.heavy[2 * b];
  const uint32_t s = w.cell_off[slot], cnt = w.cell_off[slot + 1] - s;
  const uint32_t m = sor_pow2(cnt);
  unsigned long long *P = w.pairs + w.heavy[2 * b + 1];
  const uint32_t tid = threadIdx.x, nt = blockDim.x;
  for (uint32_t r = tid; r < m; r += nt) {
    P[r] = r < cnt ? (((unsigned long long)float_to_key(w.sorted[3 * (size_t)(s + r)]) << 32) | r) : ~0ull;
    if (r < cnt) {
      w.tmp_xyz[3 * (size_t)(s + r)] = w.sorted[3 * (size_t)(s + r)];
      w.tmp_xyz[3 * (size_t)(s + r) + 1] = w.sorted[3 * (size_t)(s + r) + 1];
      w.tmp_xyz[3 * (size_t)(s + r) + 2] = w.sorted[3 * (size_t)(s + r) + 2];
      w.tmp_idx[s + r] = w.sorted_idx[s + r];
    }
  }
  __syncthreads();
  const uint32_t half = m >> 1;
  for (uint32_t kk = 2; kk <= m; kk <<= 1) {
    for (uint32_t j = kk >> 1; j > 0; j >>= 1) {
      for (uint32_t t = tid; t < half; t += nt) {
        const uint32_t a = ((t & ~(j - 1)) << 1) | (t & (j - 1));
        const uint32_t c = a | j;
        const unsigned long long x = P[a], y = P[c];
        const bool up = (a & kk) == 0;
        if ((x > y) == up) { P[a] = y; P[c] = x; }
      }
      __syncthreads();
    }
  }
  for (uint32_t r = tid; r < cnt; r += nt) {
    const uint32_t src = s + (uint32_t)(P[r] & 0xFFFFFFFFull);
    w.sorted[3 * (size_t)(s + r)] = w.tmp_xyz[3 * (size_t)src];
    w.sorted[3 * (size_t)(s + r) + 1] = w.tmp_xyz[3 * (size_t)src + 1];
    w.sorted[3 * (size_t)(s + r) + 2] = w.tmp_xyz[3 * (size_t)src + 2];
    w.sorted_idx[s + r] = w.tmp_idx[src];
  }
  if (tid == 0) w.cell_cnt[slot] = kSorSortedFlag;
}

// The k smallest squared distances of one query (a max-heap, see below).  STRIDE 1: a per-thread local array; STRIDE
// kSorThreads: one column of a [k][kSorThreads] shared-memory array (k <= kSorSharedK) -- the insertion loop is a
// chain of dependent loads and stores, and local memory competes with the candidate stream for L1.
template <int STRIDE>
struct KBest {
  double *p;
  __device__ __forceinline__ double &operator[](int t) const { return p[t * STRIDE]; }
};
constexpr int kSorSharedK = 24;

// The k smallest squared distances are kept as a binary MAX-HEAP (root = the current k-th distance).  A candidate
// that beats the root replaces it with one sift-down: at most log2(k) steps, the same few for every lane -- the
// sorted list this replaces shifted up to k entries per insertion, and a warp paid the longest lane's chain for
// every candidate any of its lanes accepted.  The ascending order the mean needs comes from one heap sort at the end.
template <class B>
__device__ __forceinline__ void kbest_sift(const B &best, int size, double v) {
  int pos = 0;
  while (true) {
    const int l = 2 * pos + 1;
    if (l >= size) break;
    const int r = l + 1;
    const double vl = best[l], vr = r < size ? best[r] : -1.0;
    const bool right = vr > vl;
    const double vc = right ? vr : vl;
    if (vc <= v) break;
    best[pos] = vc;
    pos = right ? r : l;
  }
  best[pos] = v;
}
template <class B>
__device__ __forceinline__ void kbest_push(const B &best, int k, double d2, double &kth, float &thrf) {
  kbest_sift(best, k, d2);
  kth = best[0];
  thrf = sor_filter(kth);
}
// heap -> ascending array (in place), then the sum of the square roots in ascending order
template <class B>
__device__ __forceinline__ double kbest_sorted_sqrt_sum(const B &best, int k) {
  for (int m = k; m > 1; --m) {
    const double top = best[0], last = best[m - 1];
    best[m - 1] = top;
    kbest_sift(best, m - 1, last);
  }
  double s = 0.0;
  for (int t = 0; t < k; ++t) s += sqrt(best[t]);  // ascending order, like std::accumulate over nanoflann's result
  return s;
}

// Candidates of one cell.  A float32 estimate of the squared distance (relative error < 4e-7) rejects most
// candidates for a sixth of the cost; whatever passes the (conservative) filter is evaluated exactly.
template <class B>
__device__ __forceinline__ void sor_visit_cell(const SorWs &w, uint32_t cell, const double q[3], const float qf[3],
                                               const B &best, int k, float &thrf, double &kth) {
  const uint32_t s = w.cell_off[cell], e = w.cell_off[cell + 1];
  constexpr int U = 4;  // candidates in flight per iteration (independent loads and float32 estimates)
  if (w.cell_cnt[cell] & kSorSortedFlag) {
    // Very heavy cell, points sorted by x: walk outwards from the query's x, U candidates per side and step,
    // while dx^2 can still beat the k-th distance (float32 estimate, same conservative margin as below).
    uint32_t lo = s, hi = e;
    while (lo < hi) {  // first point with x >= q.x
      const uint32_t mid = lo + ((hi - lo) >> 1);
      if (w.sorted[3 * (size_t)mid] < qf[0]) lo = mid + 1; else hi = mid;
    }
    uint32_t r = lo;   // next candidate to the right
    uint32_t l = lo;   // next candidate to the left is l - 1
    bool go_r = r < e, go_l = l > s;
    while ((go_r || go_l) && kth > 0.0) {  // k coincident points: nothing can be closer
      float p[2 * U][3];
      bool ok[2 * U];
#pragma unroll
      for (int u = 0; u < U; ++u) {  // independent loads first
        ok[u] = go_r && r + (uint32_t)u < e;
        ok[U + u] = go_l && l >= s + 1u + (uint32_t)u;
        const uint32_t jr = ok[u] ? r + (uint32_t)u : s, jl = ok[U + u] ? l - 1u - (uint32_t)u : s;
#pragma unroll
        for (int a = 0; a < 3; ++a) { p[u][a] = w.sorted[3 * (size_t)jr + a]; p[U + u][a] = w.sorted[3 * (size_t)jl + a]; }
      }
#pragma unroll
      for (int u = 0; u < 2 * U; ++u) {  // in order of growing |dx| on each side
        const bool right = u < U;
        if (!ok[u] || (right ? !go_r : !go_l)) continue;
        const float fx = qf[0] - p[u][0];
        if (fx * fx > thrf) { if (right) go_r = false; else go_l = false; continue; }
        const float fy = qf[1] - p[u][1], fz = qf[2] - p[u][2];
        const float d2f = fx * fx + fy * fy + fz * fz;
        if (d2f <= thrf) {
          const double dx = q[0] - (double)p[u][0], dy = q[1] - (double)p[u][1], dz = q[2] - (double)p[u][2];
          double d2 = dx * dx;
          d2 += dy * dy;
          d2 += dz * dz;
          if (d2 < kth) {
            kbest_push(best, k, d2, kth, thrf);
          }
        }
      }
      if (go_r) { r += U; go_r = r < e; }
      if (go_l) { l = l >= s + (uint32_t)U ? l - (uint32_t)U : s; go_l = l > s; }
    }
    return;
  }
  for (uint32_t j0 = s; j0 < e && kth > 0.0; j0 += U) {  // (k coincident points end the search)
    float p[U][3], d2f[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const uint32_t j = min(j0 + (uint32_t)u, e - 1u);  // the tail repeats the last candidate (harmless: not < kth twice)
#pragma unroll
      for (int a = 0; a < 3; ++a) p[u][a] = w.sorted[3 * (size_t)j + a];
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const float fx = qf[0] - p[u][0], fy = qf[1] - p[u][1], fz = qf[2] - p[u][2];
      d2f[u] = fx * fx + fy * fy + fz * fz;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (j0 + (uint32_t)u >= e || d2f[u] > thrf) continue;
      const double dx = q[0] - (double)p[u][0], dy = q[1] - (double)p[u][1], dz = q[2] - (double)p[u][2];
      double d2 = dx * dx;   // nanoflann L2_Simple: result += diff * diff, axis by axis (no contraction: --fmad=false)
      d2 += dy * dy;
      d2 += dz * dz;
      if (d2 < kth) {
        kbest_push(best, k, d2, kth, thrf);
      }
    }
  }
}

// a neighbour cell by key: one hash probe; most cells of a shell do not exist
template <class B>
__device__ __forceinline__ void sor_visit_key(const SorWs &w, unsigned long long key, const double q[3], const float qf[3],
                                              const B &best, int k, float &thrf, double &kth) {
  uint32_t slot;
  if (sor_find(w, key, &slot)) sor_visit_cell(w, slot, q, qf, best, k, thrf, kth);
}

// Queries run in CELL order (thread j owns the j-th sorted point): the lanes of a warp then share their
// query cell, walk the same candidate lists with the same trip counts and read the same addresses.
template <bool SHARED>
__global__ void __launch_bounds__(kSorThreads, 4) sor_query_kernel(SorWs w, int nb_neighbors) {
  extern __shared__ double s_best[];   // SHARED: [k][kSorThreads]
  const SorHeader *h = w.hdr;
  const uint32_t n = h->n;
  const uint32_t j = blockIdx.x * (uint32_t)kSorThreads + threadIdx.x;
  if (j >= n) return;
  const uint32_t i = w.sorted_idx[j];
  const int k = (int)min((uint32_t)nb_neighbors, n);
  double loc[SHARED ? 1 : kSorMaxK];
  const KBest<SHARED ? kSorThreads : 1> best{SHARED ? s_best + threadIdx.x : loc};
  for (int t = 0; t < k; ++t) best[t] = __longlong_as_double(0x7FF0000000000000ll);
  double kth = __longlong_as_double(0x7FF0000000000000ll);
  const float qf[3] = {w.sorted[3 * (size_t)j], w.sorted[3 * (size_t)j + 1], w.sorted[3 * (size_t)j + 2]};
  const double q[3] = {(double)qf[0], (double)qf[1], (double)qf[2]};
  float thrf = __int_as_float(0x7F800000);
  const int32_t nx = h->dim[0], ny = h->dim[1], nz = h->dim[2];
  const uint32_t cell = w.pt_cell[i];
  const unsigned long long ckey = w.keys[cell];
  const int32_t cm = (1 << kSorCoordBits) - 1;
  const int32_t c0 = (int32_t)(ckey >> (2 * kSorCoordBits)) & cm, c1 = (int32_t)(ckey >> kSorCoordBits) & cm,
                c2 = (int32_t)ckey & cm;
  const int32_t c[3] = {c0, c1, c2};
  // distances from the query to the faces of its own cell (0 if rounding put it outside)
  double dlo[3], dhi[3];
  int32_t rmax = 0;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const double lo = h->mn[a] + (double)c[a] * h->h;
    dlo[a] = fmax(q[a] - lo, 0.0);
    dhi[a] = fmax(lo + h->h - q[a], 0.0);
    rmax = max(rmax, max(c[a], h->dim[a] - 1 - c[a]));
  }
  sor_visit_cell(w, cell, q, qf, best, k, thrf, kth);
  const int32_t dim[3] = {nx, ny, nz};
  for (int32_t R = 1; R <= rmax; ++R) {
    // Unvisited points lie beyond a face of the block of radius R - 1 that is still inside the grid:
    // at least (R - 1) * h + (distance to the own cell's face on that side) away.
    double reach = __longlong_as_double(0x7FF0000000000000ll);
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      if (c[a] - R >= 0) reach = fmin(reach, (double)(R - 1) * h->h + dlo[a]);
      if (c[a] + R <= dim[a] - 1) reach = fmin(reach, (double)(R - 1) * h->h + dhi[a]);
    }
    reach -= h->slack;
    if ((reach > 0.0 && kth <= reach * reach) || kth == 0.0) break;
    // shell of Chebyshev radius R, clipped to the grid, as six slabs (no cell is visited twice):
    //   x faces: a0 = c0 -+ R, full (a1, a2) range;  y faces: a1 = c1 -+ R, a0 interior;  z faces: a0, a1 interior
    const int32_t x0 = max(c0 - R, 0), x1 = min(c0 + R, nx - 1);
    const int32_t y0 = max(c1 - R, 0), y1 = min(c1 + R, ny - 1);
    const int32_t z0 = max(c2 - R, 0), z1 = min(c2 + R, nz - 1);
    const int32_t xi0 = max(c0 - R + 1, 0), xi1 = min(c0 + R - 1, nx - 1);  // interior ranges
    const int32_t yi0 = max(c1 - R + 1, 0), yi1 = min(c1 + R - 1, ny - 1);
    for (int side = 0; side < 2; ++side) {
      const int32_t a0 = side ? c0 + R : c0 - R;
      if (a0 < 0 || a0 >= nx) continue;
      for (int32_t a1 = y0; a1 <= y1; ++a1)
        for (int32_t a2 = z0; a2 <= z1; ++a2) sor_visit_key(w, sor_key(a0, a1, a2), q, qf, best, k, thrf, kth);
    }
    for (int side = 0; side < 2; ++side) {
      const int32_t a1 = side ? c1 + R : c1 - R;
      if (a1 < 0 || a1 >= ny) continue;
      for (int32_t a0 = xi0; a0 <= xi1; ++a0)
        for (int32_t a2 = z0; a2 <= z1; ++a2) sor_visit_key(w, sor_key(a0, a1, a2), q, qf, best, k, thrf, kth);
    }
    for (int side = 0; side < 2; ++side) {
      const int32_t a2 = side ? c2 + R : c2 - R;
      if (a2 < 0 || a2 >= nz) continue;
      for (int32_t a0 = xi0; a0 <= xi1; ++a0)
        for (int32_t a1 = yi0; a1 <= yi1; ++a1) sor_visit_key(w, sor_key(a0, a1, a2), q, qf, best, k, thrf, kth);
    }
  }
  w.avg[i] = kbest_sorted_sqrt_sum(best, k) / (double)k;
}

// cloud mean, Bessel-corrected standard deviation and the threshold.  Two passes (sum, then squared
// deviations); each pass: kSorStatBlocks CTAs write one partial each (fixed assignment of rows to threads and
// a fixed tree inside the CTA), then one thread adds the partials in order: deterministic.
constexpr int kSorStatBlocks = 256;
__global__ void __launch_bounds__(1024) sor_partial_kernel(SorWs w, int pass, double *partial) {
  __shared__ double s_red[1024];
  const SorHeader *h = w.hdr;
  const uint32_t n = h->n;
  const int tid = threadIdx.x;
  const double mean = h->cloud_mean;
  double acc = 0.0;
  for (uint32_t i = blockIdx.x * 1024u + tid; i < n; i += (uint32_t)kSorStatBlocks * 1024u) {
    const double a = w.avg[i];
    if (a > 0.0) acc += pass == 0 ? a : (a - mean) * (a - mean);
  }
  s_red[tid] = acc;
  __syncthreads();
  for (int s = 512; s > 0; s >>= 1) {
    if (tid < s) s_red[tid] += s_red[tid + s];
    __syncthreads();
  }
  if (tid == 0) partial[blockIdx.x] = s_red[0];
}
__global__ void sor_finish_kernel(SorWs w, int pass, const double *partial, double std_ratio, double *stats) {
  if (threadIdx.x != 0) return;
  SorHeader *h = w.hdr;
  const uint32_t n = h->n;
  double t = 0.0;
  for (int b = 0; b < kSorStatBlocks; ++b) t += partial[b];
  if (pass == 0) {
    h->cloud_mean = n > 0 ? t / (double)n : 0.0;
  } else {
    h->std_dev = sqrt(t / ((double)n - 1.0));
    h->thr = h->cloud_mean + std_ratio * h->std_dev;
    if (stats) { stats[0] = h->cloud_mean; stats[1] = h->std_dev; stats[2] = h->thr; stats[3] = (double)n; }
  }
}

__device__ __forceinline__ bool sor_keep(const SorWs &w, uint32_t i) {
  const double a = w.avg[i];
  return a > 0.0 && a < w.hdr->thr;
}

__global__ void __launch_bounds__(kSorThreads) sor_keep_count_kernel(SorWs w) {
  __shared__ uint32_t s_warp[kSorThreads / 32];
  const uint32_t n = w.hdr->n;
  if (blockIdx.x * (uint32_t)kSorThreads >= n) return;
  const uint32_t i = blockIdx.x * (uint32_t)kSorThreads + threadIdx.x;
  uint32_t total;
  block_excl_scan((i < n && sor_keep(w, i)) ? 1u : 0u, s_warp, &total);
  if (threadIdx.x == 0) w.tile_cnt[blockIdx.x] = total;
}

__global__ void __launch_bounds__(kSorScanThreads) sor_tile_scan_kernel(SorWs w, uint32_t *out_count) {
  __shared__ uint32_t s_warp[32];
  __shared__ uint32_t s_carry;
  const uint32_t nt = (w.hdr->n + kSorThreads - 1) / kSorThreads;
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  for (uint32_t base = 0; base < nt; base += kSorScanThreads) {
    const uint32_t i = base + threadIdx.x;
    const uint32_t v = i < nt ? w.tile_cnt[i] : 0u;
    uint32_t total;
    const uint32_t ex = block_excl_scan(v, s_warp, &total);
    if (i < nt) w.tile_cnt[i] = s_carry + ex;
    __syncthreads();
    if (threadIdx.x == 0) s_carry += total;
    __syncthreads();
  }
  if (threadIdx.x == 0) *out_count = s_carry;
}

__global__ void __launch_bounds__(kSorThreads) sor_compact_kernel(SorWs w, const float *xyz, const float *rgb, float *oxyz,
                                                                  float *orgb, uint32_t *oindex) {
  __shared__ uint32_t s_warp[kSorThreads / 32];
  const uint32_t n = w.hdr->n;
  if (blockIdx.x * (uint32_t)kSorThreads >= n) return;
  const uint32_t i = blockIdx.x * (uint32_t)kSorThreads + threadIdx.x;
  const bool keep = i < n && sor_keep(w, i);
  uint32_t total;
  const uint32_t ex = block_excl_scan(keep ? 1u : 0u, s_warp, &total);
  if (!keep) return;
  const size_t dst = (size_t)w.tile_cnt[blockIdx.x] + ex;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    oxyz[3 * dst + k] = __ldg(xyz + 3 * (size_t)i + k);
    if (orgb) orgb[3 * dst + k] = __ldg(rgb + 3 * (size_t)i + k);
  }
  if (oindex) oindex[dst] = i;
}

int sor_grid_build(const SorWs &w, const float *d_xyz, const uint32_t *d_count, const float *d_bounds,
                   uint32_t capacity_rows, cudaStream_t st) {
  const uint32_t row_blocks = (capacity_rows + kSorThreads - 1) / kSorThreads;
  const uint32_t stride_blocks = min(row_blocks, 148u * 16u);
  const uint32_t cell_blocks = w.cap / kSorScanThreads + 1;
  sor_begin_kernel<<<1, 32, 0, st>>>(w, d_count, d_bounds);
  D2PC_CHECK_LAUNCH();
  for (int t = 0; t < kSorTrials; ++t) {  // occupied cells for every candidate cell size
    sor_clear_kernel<<<148 * 8, 256, 0, st>>>(w);
    D2PC_CHECK_LAUNCH();
    sor_trial_kernel<<<stride_blocks, kSorThreads, 0, st>>>(w, d_xyz, t);
    D2PC_CHECK_LAUNCH();
  }
  const char *occ_env = getenv("D2PC_SOR_OCC");  // measurement aid
  sor_choose_kernel<<<1, 32, 0, st>>>(w, occ_env ? atof(occ_env) : kSorTargetOcc);
  D2PC_CHECK_LAUNCH();
  sor_clear_kernel<<<148 * 8, 256, 0, st>>>(w);
  D2PC_CHECK_LAUNCH();
  sor_count_kernel<<<stride_blocks, kSorThreads, 0, st>>>(w, d_xyz);
  D2PC_CHECK_LAUNCH();
  sor_scan1_kernel<<<cell_blocks, kSorScanThreads, 0, st>>>(w);
  D2PC_CHECK_LAUNCH();
  sor_scan2_kernel<<<1, kSorScanThreads, 0, st>>>(w);
  D2PC_CHECK_LAUNCH();
  sor_scan3_kernel<<<cell_blocks, kSorScanThreads, 0, st>>>(w);
  D2PC_CHECK_LAUNCH();
  sor_scatter_kernel<<<stride_blocks, kSorThreads, 0, st>>>(w, d_xyz);
  D2PC_CHECK_LAUNCH();
  sor_heavy_list_kernel<<<148 * 8, 256, 0, st>>>(w);
  D2PC_CHECK_LAUNCH();
  sor_heavy_offsets_kernel<<<1, 32, 0, st>>>(w);
  D2PC_CHECK_LAUNCH();
  sor_heavy_sort_kernel<<<kSorMaxHeavy, 1024, 0, st>>>(w);
  D2PC_CHECK_LAUNCH();
  return D2PC_OK;
}

int sor_grid_build_fixed(const SorWs &w, const float *d_xyz, const uint32_t *d_count, const float *d_bounds, double cs,
                         uint32_t capacity_rows, uint32_t *d_err, cudaStream_t st) {
  const uint32_t row_blocks = (capacity_rows + kSorThreads - 1) / kSorThreads;
  const uint32_t stride_blocks = min(row_blocks, 148u * 16u);
  const uint32_t cell_blocks = w.cap / kSorScanThreads + 1;
  sor_fixed_begin_kernel<<<1, 32, 0, st>>>(w, d_count, d_bounds, cs, d_err);
  D2PC_CHECK_LAUNCH();
  sor_clear_kernel<<<148 * 8, 256, 0, st>>>(w);
  D2PC_CHECK_LAUNCH();
  sor_count_kernel<<<stride_blocks, kSorThreads, 0, st>>>(w, d_xyz);
  D2PC_CHECK_LAUNCH();
  sor_scan1_kernel<<<cell_blocks, kSorScanThreads, 0, st>>>(w);
  D2PC_CHECK_LAUNCH();
  sor_scan2_kernel<<<1, kSorScanThreads, 0, st>>>(w);
  D2PC_CHECK_LAUNCH();
  sor_scan3_kernel<<<cell_blocks, kSorScanThreads, 0, st>>>(w);
  D2PC_CHECK_LAUNCH();
  sor_scatter_kernel<<<stride_blocks, kSorThreads, 0, st>>>(w, d_xyz);
  D2PC_CHECK_LAUNCH();
  return D2PC_OK;
}

int sor_compact(const SorWs &w, const float *d_xyz, const float *d_rgb, float *d_out_xyz, float *d_out_rgb,
                uint32_t *d_out_index, uint32_t *d_out_count, uint32_t capacity_rows, cudaStream_t st) {
  const uint32_t row_blocks = (capacity_rows + kSorThreads - 1) / kSorThreads;
  sor_keep_count_kernel<<<row_blocks, kSorThreads, 0, st>>>(w);
  D2PC_CHECK_LAUNCH();
  sor_tile_scan_kernel<<<1, kSorScanThreads, 0, st>>>(w, d_out_count);
  D2PC_CHECK_LAUNCH();
  sor_compact_kernel<<<row_blocks, kSorThreads, 0, st>>>(w, d_xyz, d_rgb, d_out_xyz, d_out_rgb, d_out_index);
  D2PC_CHECK_LAUNCH();
  return D2PC_OK;
}

}  // namespace d2pc

using namespace d2pc;

extern "C" int d2pc_sor_scratch_bytes(uint32_t capacity_rows, size_t *bytes) {
  if (!bytes || capacity_rows == 0) return D2PC_ERR_INVALID_ARGUMENT;
  *bytes = sor_ws_bytes(capacity_rows);
  return D2PC_OK;
}

extern "C" int d2pc_sor_enqueue(const float *d_xyz, const float *d_rgb, const uint32_t *d_count, uint32_t capacity_rows,
                                const float *d_bounds, int32_t nb_neighbors, double std_ratio, void *d_scratch,
                                size_t scratch_bytes, float *d_out_xyz, float *d_out_rgb, uint32_t *d_out_index,
                                uint32_t *d_out_count, double *d_stats, void *stream) {
  if (!d_xyz || !d_count || !d_bounds || !d_scratch || !d_out_xyz || !d_out_count) return D2PC_ERR_INVALID_ARGUMENT;
  if ((d_out_rgb != nullptr) != (d_rgb != nullptr)) return D2PC_ERR_INVALID_ARGUMENT;
  if (capacity_rows == 0 || nb_neighbors < 1 || nb_neighbors > kSorMaxK || !(std_ratio > 0.0)) return D2PC_ERR_INVALID_ARGUMENT;
  if (((uintptr_t)d_scratch & 255u) != 0) return D2PC_ERR_INVALID_ARGUMENT;
  if (scratch_bytes < sor_ws_bytes(capacity_rows)) return D2PC_ERR_WORKSPACE_TOO_SMALL;
  cudaStream_t st = (cudaStream_t)stream;
  SorWs w = sor_ws(d_scratch, capacity_rows);
  const uint32_t row_blocks = (capacity_rows + kSorThreads - 1) / kSorThreads;
  const int rc = sor_grid_build(w, d_xyz, d_count, d_bounds, capacity_rows, st);
  if (rc != D2PC_OK) return rc;
  if (nb_neighbors <= kSorSharedK) {
    const size_t smem = (size_t)nb_neighbors * kSorThreads * sizeof(double);   // <= 48 KB
    sor_query_kernel<true><<<row_blocks, kSorThreads, smem, st>>>(w, nb_neighbors);
  } else {
    sor_query_kernel<false><<<row_blocks, kSorThreads, 0, st>>>(w, nb_neighbors);
  }
  D2PC_CHECK_LAUNCH();
  double *partial = reinterpret_cast<double *>(w.blk_sum);  // the cell scan is done with it
  for (int pass = 0; pass < 2; ++pass) {
    sor_partial_kernel<<<kSorStatBlocks, 1024, 0, st>>>(w, pass, partial);
    D2PC_CHECK_LAUNCH();
    sor_finish_kernel<<<1, 32, 0, st>>>(w, pass, partial, std_ratio, d_stats);
    D2PC_CHECK_LAUNCH();
  }
  return sor_compact(w, d_xyz, d_rgb, d_out_xyz, d_out_rgb, d_out_index, d_out_count, capacity_rows, st);
}
