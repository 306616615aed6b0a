// d2pc_cluster.cu -- row f5: density clustering of a point cloud, Open3D ClusterDBSCAN and RemoveRadiusOutliers
// (spec: oracle/d2pc_cluster_oracle.py; Open3D itself is not installed: parity unpinned).
//   neighbours  j of i when d2(i, j) < eps^2, d2 summed axis by axis in float64 (--fmad=false), i itself included
//   radius      keep i iff |N(i)| > nb_points, kept rows in input order
//   DBSCAN      core iff |N(i)| >= min_points; clusters = components of the cores, numbered by their lowest core row;
//               a non-core row takes the lowest cluster among its core neighbours, else -1
//
// The grid is statistical outlier removal's (d2pc_grid.cuh) with the cell side cs = eps / 2 * (1 + 2^-20):
//   * two rows of one cell are within sqrt(3) * cs = 0.866 * eps of each other, far inside eps whatever the
//     rounding of the cell coordinates (relative 2^-50), so a cell's rows are all neighbours of each other;
//   * a neighbour differs by less than eps / cs = 2 - 2^-19 cells per axis, so it lies in the 5 x 5 x 5 block of
//     cells around a row's own cell (the coordinates' rounding error is ~2^-31 cells, the margin 2^-19);
//   * both need unclamped coordinates: an axis that needs kSorCellLimit cells or more is refused (error word).
// Every occupied cell keeps the tight box of its members (float keys at the cell's first sorted row).  A cell whose
// box is at least eps away (with a relative margin kBoxMargin, far above the ~2^-50 error of the float64 box and
// point distances) is skipped; a cell whose box lies wholly within eps (same margin) is taken whole.  That keeps the
// rows near the clump of clipped pixels (thousands of rows in a box ~1e-7 wide) from walking it row by row.
//
//   box      per cell: min / max of the members (warp-segmented, one atomic per warp run); non-finite rows
//   count    |N(i)| up to the threshold: own cell whole, then the 124 others; core flag by sorted row, and
//            parent[i] = i for a core, kCompNone otherwise
//   rep      per cell: its lowest core row (warp-segmented atomicMin)
//   unite1   every core of a cell under the cell's lowest core (no distance test: they are neighbours)
//   unite2   every core against the cells of the 62 positive offsets: stops at the first core within eps, and
//            skips a cell whose lowest core is already in its set (all the cores of a cell are one set)
//   number   roots per tile, tile scan (d2pc_scan.cuh), cluster id of every root; labels of the cores
//   border   a non-core row: the lowest cluster among the cells holding a core neighbour (one cluster per cell)
//   sizes    rows per cluster (one atomic per warp group of equal labels)
//   keep     the decision as avg 1 / 0 with threshold 2, then statistical outlier removal's ordered compaction
#include <cuda_runtime.h>
#include "d2pc_grid.cuh"
#include "d2pc_scan.cuh"
#include "d2pc_components.h"

namespace d2pc {

constexpr int kClThreads = 256;
constexpr double kBoxMargin = 1e-12;

struct ClusterWs {
  SorWs g;
  uint8_t *core;     // [N] by sorted row
  uint32_t *box;     // [6][N] float keys of min x, y, z, max x, y, z of every cell, at its first sorted row
  uint32_t *rep;     // [N] lowest core (source row) of every cell, at its first sorted row; kCompNone: no core
  uint32_t *parent;  // [N] union-find forest by source row (kCompNone: not a core)
  uint32_t *cid;     // [N] cluster id of every root
  uint32_t cap_rows;
};

inline size_t cluster_ws_bytes(uint32_t n) {
  return sor_ws_bytes(n) + align_up(n, 256) + align_up((size_t)n * 24, 256) + 3 * align_up((size_t)n * 4, 256);
}
inline ClusterWs cluster_ws(void *base, uint32_t n) {
  ClusterWs w;
  w.g = sor_ws(base, n);
  char *p = (char *)base + sor_ws_bytes(n);
  w.core = (uint8_t *)p;     p += align_up(n, 256);
  w.box = (uint32_t *)p;     p += align_up((size_t)n * 24, 256);
  w.rep = (uint32_t *)p;     p += align_up((size_t)n * 4, 256);
  w.parent = (uint32_t *)p;  p += align_up((size_t)n * 4, 256);
  w.cid = (uint32_t *)p;
  w.cap_rows = n;
  return w;
}

__device__ __forceinline__ double cl_d2(const double q[3], const float *p) {
  const double dx = q[0] - (double)p[0], dy = q[1] - (double)p[1], dz = q[2] - (double)p[2];
  double d2 = dx * dx;
  d2 += dy * dy;
  d2 += dz * dz;
  return d2;
}

// the cell coordinates of a slot, from its key
__device__ __forceinline__ void cl_coords(const SorWs &g, uint32_t slot, int32_t c[3]) {
  const unsigned long long key = g.keys[slot];
  const int32_t cm = (1 << kSorCoordBits) - 1;
  c[0] = (int32_t)(key >> (2 * kSorCoordBits)) & cm;
  c[1] = (int32_t)(key >> kSorCoordBits) & cm;
  c[2] = (int32_t)key & cm;
}

// slot of the cell at c + (dx, dy, dz), false when it is outside the grid or empty
__device__ __forceinline__ bool cl_cell(const SorWs &g, const int32_t c[3], int dx, int dy, int dz, uint32_t *slot) {
  const int32_t a = c[0] + dx, b = c[1] + dy, e = c[2] + dz;
  const SorHeader *h = g.hdr;
  if (a < 0 || b < 0 || e < 0 || a >= h->dim[0] || b >= h->dim[1] || e >= h->dim[2]) return false;
  return sor_find(g, sor_key(a, b, e), slot);
}

// -1: every member of the cell at first sorted row s is at least eps away; 1: every member is within eps; 0: test
__device__ __forceinline__ int cl_box_test(const ClusterWs &w, uint32_t s, const double q[3], double eps2) {
  const uint32_t N = w.cap_rows;
  double gap = 0.0, far = 0.0;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const double lo = (double)key_to_float(w.box[a * N + s]), hi = (double)key_to_float(w.box[(3 + a) * N + s]);
    const double g = fmax(fmax(lo - q[a], q[a] - hi), 0.0), f = fmax(q[a] - lo, hi - q[a]);
    gap += g * g;
    far += f * f;
  }
  if (gap >= eps2 * (1.0 + kBoxMargin)) return -1;
  if (far <= eps2 * (1.0 - kBoxMargin)) return 1;
  return 0;
}

__device__ __forceinline__ void cl_fail(uint32_t *counts, uint32_t bit) { atomicOr(counts + 1, bit); }

// Inclusive segmented min / max over the lanes of a warp whose `seg` values are equal and contiguous; `start` is the
// first lane of the caller's segment.
__device__ __forceinline__ uint32_t seg_min(uint32_t v, int start) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t y = __shfl_up_sync(0xffffffffu, v, d);
    if (lane - d >= start) v = min(v, y);
  }
  return v;
}
__device__ __forceinline__ uint32_t seg_max(uint32_t v, int start) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t y = __shfl_up_sync(0xffffffffu, v, d);
    if (lane - d >= start) v = max(v, y);
  }
  return v;
}
// segments of equal `seg` (the cell's first sorted row); returns the first lane of this lane's segment, *tail = the
// lane is the last of its segment
__device__ __forceinline__ int seg_start(uint32_t seg, bool *tail) {
  const int lane = threadIdx.x & 31;
  const uint32_t prev = __shfl_up_sync(0xffffffffu, seg, 1);
  const uint32_t heads = __ballot_sync(0xffffffffu, lane == 0 || prev != seg);
  *tail = lane == 31 || ((heads >> (lane + 1)) & 1u);
  return 31 - __clz(heads & (0xFFFFFFFFu >> (31 - lane)));
}

// box of every cell; non-finite rows
__global__ void __launch_bounds__(kClThreads) cl_box_kernel(ClusterWs w, uint32_t *counts) {
  const SorWs &g = w.g;
  const uint32_t n = g.hdr->n;
  const uint32_t j = blockIdx.x * kClThreads + threadIdx.x;
  if (blockIdx.x * kClThreads >= n) return;   // whole warps stay together below (this kernel sets the error word)
  const bool live = j < n;
  uint32_t s = 0xFFFFFFFFu;
  float p[3] = {0.0f, 0.0f, 0.0f};
  if (live) {
    s = g.cell_off[g.pt_cell[g.sorted_idx[j]]];
#pragma unroll
    for (int a = 0; a < 3; ++a) p[a] = g.sorted[3 * (size_t)j + a];
    if (!(isfinite(p[0]) && isfinite(p[1]) && isfinite(p[2]))) cl_fail(counts, D2PC_CLUSTER_ERR_NONFINITE);
  }
  bool tail;
  const int start = seg_start(s, &tail);
  const uint32_t N = w.cap_rows;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const uint32_t k = float_to_key(p[a]);
    const uint32_t lo = seg_min(k, start), hi = seg_max(k, start);
    if (live && tail) {
      atomicMin(&w.box[a * N + s], lo);
      atomicMax(&w.box[(3 + a) * N + s], hi);
    }
  }
}

// |N(i)| up to thr (a row stops as soon as it gets there): core flag by sorted row, parent by source row
__global__ void __launch_bounds__(kClThreads) cl_count_kernel(ClusterWs w, double eps2, uint32_t thr, uint32_t *counts) {
  const SorWs &g = w.g;
  const uint32_t n = g.hdr->n;
  const uint32_t j = blockIdx.x * kClThreads + threadIdx.x;
  if (j >= n || counts[1]) return;
  const uint32_t i = g.sorted_idx[j], slot = g.pt_cell[i];
  const double q[3] = {(double)g.sorted[3 * (size_t)j], (double)g.sorted[3 * (size_t)j + 1],
                       (double)g.sorted[3 * (size_t)j + 2]};
  int32_t c[3];
  cl_coords(g, slot, c);
  uint32_t cnt = g.cell_off[slot + 1] - g.cell_off[slot];   // the own cell, whole
  for (int o = 0; o < 125 && cnt < thr; ++o) {
    const int dx = o / 25 - 2, dy = (o / 5) % 5 - 2, dz = o % 5 - 2;
    uint32_t sl;
    if ((dx | dy | dz) == 0 || !cl_cell(g, c, dx, dy, dz, &sl)) continue;
    const uint32_t s = g.cell_off[sl], e = g.cell_off[sl + 1];
    const int t = cl_box_test(w, s, q, eps2);
    if (t < 0) continue;
    if (t > 0) { cnt += e - s; continue; }
    for (uint32_t m = s; m < e && cnt < thr; ++m) cnt += cl_d2(q, g.sorted + 3 * (size_t)m) < eps2 ? 1u : 0u;
  }
  const bool core = cnt >= thr;
  w.core[j] = core ? 1 : 0;
  w.parent[i] = core ? i : kCompNone;
}

// lowest core (source row) of every cell
__global__ void __launch_bounds__(kClThreads) cl_rep_kernel(ClusterWs w, const uint32_t *counts) {
  const SorWs &g = w.g;
  const uint32_t n = g.hdr->n;
  const uint32_t j = blockIdx.x * kClThreads + threadIdx.x;
  if (blockIdx.x * kClThreads >= n || counts[1]) return;
  const bool live = j < n;
  uint32_t s = 0xFFFFFFFFu, v = kCompNone;
  if (live) {
    const uint32_t i = g.sorted_idx[j];
    s = g.cell_off[g.pt_cell[i]];
    if (w.core[j]) v = i;
  }
  bool tail;
  const int start = seg_start(s, &tail);
  v = seg_min(v, start);
  if (live && tail && v != kCompNone) atomicMin(&w.rep[s], v);
}

// every core of a cell under the cell's lowest core
__global__ void __launch_bounds__(kClThreads) cl_unite_cell_kernel(ClusterWs w, uint32_t *counts) {
  const SorWs &g = w.g;
  const uint32_t n = g.hdr->n;
  const uint32_t j = blockIdx.x * kClThreads + threadIdx.x;
  if (j >= n || counts[1] || !w.core[j]) return;
  const uint32_t i = g.sorted_idx[j];
  const uint32_t r = w.rep[g.cell_off[g.pt_cell[i]]];
  if (r != i && comp_unite(w.parent, i, r, n) == kCompFail) cl_fail(counts, D2PC_CLUSTER_ERR_BOUND);
}

// every core against the cells at the 62 positive offsets of the 5 x 5 x 5 block (each unordered cell pair once)
__global__ void __launch_bounds__(kClThreads) cl_unite_near_kernel(ClusterWs w, double eps2, uint32_t *counts) {
  const SorWs &g = w.g;
  const uint32_t n = g.hdr->n;
  const uint32_t j = blockIdx.x * kClThreads + threadIdx.x;
  if (j >= n || counts[1] || !w.core[j]) return;
  const uint32_t i = g.sorted_idx[j], slot = g.pt_cell[i];
  const uint32_t own = w.rep[g.cell_off[slot]];
  const double q[3] = {(double)g.sorted[3 * (size_t)j], (double)g.sorted[3 * (size_t)j + 1],
                       (double)g.sorted[3 * (size_t)j + 2]};
  int32_t c[3];
  cl_coords(g, slot, c);
  for (int o = 63; o < 125; ++o) {   // offsets after (0, 0, 0) in (dx, dy, dz) order
    const int dx = o / 25 - 2, dy = (o / 5) % 5 - 2, dz = o % 5 - 2;
    uint32_t sl;
    if (!cl_cell(g, c, dx, dy, dz, &sl)) continue;
    const uint32_t s = g.cell_off[sl], e = g.cell_off[sl + 1];
    const uint32_t r = w.rep[s];
    if (r == kCompNone) continue;
    const int t = cl_box_test(w, s, q, eps2);
    if (t < 0) continue;
    const uint32_t ra = comp_find(w.parent, own, n), rb = comp_find(w.parent, r, n);
    if (ra == kCompFail || rb == kCompFail) { cl_fail(counts, D2PC_CLUSTER_ERR_BOUND); return; }
    if (ra == rb) continue;
    uint32_t hit = kCompNone;
    if (t > 0) {
      hit = r;
    } else {
      for (uint32_t m = s; m < e; ++m) {
        if (w.core[m] && cl_d2(q, g.sorted + 3 * (size_t)m) < eps2) { hit = g.sorted_idx[m]; break; }
      }
    }
    if (hit != kCompNone && comp_unite(w.parent, i, hit, n) == kCompFail) {
      cl_fail(counts, D2PC_CLUSTER_ERR_BOUND);
      return;
    }
  }
}

// roots per tile of kClThreads source rows (every tile of the capacity writes its count)
__global__ void __launch_bounds__(kClThreads) cl_root_count_kernel(ClusterWs w, const uint32_t *counts) {
  __shared__ uint32_t s_warp[kClThreads / 32];
  const uint32_t n = w.g.hdr->n;
  const uint32_t i = blockIdx.x * kClThreads + threadIdx.x;
  const bool root = i < n && !counts[1] && w.parent[i] == i;
  uint32_t total;
  tile_excl_scan(root ? 1u : 0u, s_warp, &total);
  if (threadIdx.x == 0) w.g.tile_cnt[blockIdx.x] = total;
}
__global__ void __launch_bounds__(kClThreads) cl_root_id_kernel(ClusterWs w, const uint32_t *counts) {
  __shared__ uint32_t s_warp[kClThreads / 32];
  const uint32_t n = w.g.hdr->n;
  const uint32_t i = blockIdx.x * kClThreads + threadIdx.x;
  if (blockIdx.x * kClThreads >= n || counts[1]) return;
  const bool root = i < n && w.parent[i] == i;
  uint32_t total;
  const uint32_t ex = tile_excl_scan(root ? 1u : 0u, s_warp, &total);
  if (root) w.cid[i] = w.g.tile_cnt[blockIdx.x] + ex;
}
// labels of the cores (-1 for the rest, until the border pass)
__global__ void __launch_bounds__(kClThreads) cl_core_label_kernel(ClusterWs w, int32_t *labels, uint32_t *counts) {
  const uint32_t n = w.g.hdr->n;
  const uint32_t i = blockIdx.x * kClThreads + threadIdx.x;
  if (i >= n || counts[1]) return;
  if (w.parent[i] == kCompNone) { labels[i] = -1; return; }
  const uint32_t r = comp_find(w.parent, i, n);
  if (r == kCompFail) { cl_fail(counts, D2PC_CLUSTER_ERR_BOUND); return; }
  labels[i] = (int32_t)w.cid[r];
}

// a non-core row: the lowest cluster among its core neighbours; all the cores of a cell share one cluster, so a
// cell is skipped when its cluster is not lower than the best so far, and left at the first core within eps
__global__ void __launch_bounds__(kClThreads) cl_border_kernel(ClusterWs w, double eps2, int32_t *labels,
                                                               const uint32_t *counts) {
  const SorWs &g = w.g;
  const uint32_t n = g.hdr->n;
  const uint32_t j = blockIdx.x * kClThreads + threadIdx.x;
  if (j >= n || counts[1] || w.core[j]) return;
  const uint32_t i = g.sorted_idx[j], slot = g.pt_cell[i];
  const double q[3] = {(double)g.sorted[3 * (size_t)j], (double)g.sorted[3 * (size_t)j + 1],
                       (double)g.sorted[3 * (size_t)j + 2]};
  int32_t c[3];
  cl_coords(g, slot, c);
  int32_t best = 0x7FFFFFFF;
  for (int o = 0; o < 125; ++o) {
    const int dx = o / 25 - 2, dy = (o / 5) % 5 - 2, dz = o % 5 - 2;
    uint32_t sl;
    if (!cl_cell(g, c, dx, dy, dz, &sl)) continue;
    const uint32_t s = g.cell_off[sl], e = g.cell_off[sl + 1];
    const uint32_t r = w.rep[s];
    if (r == kCompNone) continue;
    const int32_t lab = labels[r];
    if (lab >= best) continue;
    if ((dx | dy | dz) == 0) { best = lab; continue; }   // the own cell: every member is a neighbour
    const int t = cl_box_test(w, s, q, eps2);
    if (t < 0) continue;
    bool hit = t > 0;
    for (uint32_t m = s; m < e && !hit; ++m) hit = w.core[m] && cl_d2(q, g.sorted + 3 * (size_t)m) < eps2;
    if (hit) best = lab;
  }
  labels[i] = best == 0x7FFFFFFF ? -1 : best;
}

// rows per cluster: the lanes of a warp with equal labels add once
__global__ void __launch_bounds__(kClThreads) cl_sizes_kernel(ClusterWs w, const int32_t *labels, uint32_t *sizes,
                                                              const uint32_t *counts) {
  const uint32_t n = w.g.hdr->n;
  const uint32_t i = blockIdx.x * kClThreads + threadIdx.x;
  if (blockIdx.x * kClThreads >= n || counts[1]) return;
  const int32_t lab = i < n ? labels[i] : -1;
  const uint32_t group = __match_any_sync(0xffffffffu, lab);
  if (lab >= 0 && (threadIdx.x & 31) == (uint32_t)(__ffs(group) - 1)) atomicAdd(&sizes[lab], (uint32_t)__popc(group));
}

// the keep decision as statistical outlier removal's compaction reads it: avg 1 (kept) or 0, threshold 2
__global__ void __launch_bounds__(kClThreads) cl_keep_kernel(ClusterWs w, const int32_t *labels, const uint32_t *sizes,
                                                             uint32_t min_size, const uint32_t *counts) {
  const uint32_t n = w.g.hdr->n;
  const uint32_t i = blockIdx.x * kClThreads + threadIdx.x;
  if (i == 0) w.g.hdr->thr = 2.0;
  if (i >= n) return;
  bool keep = false;
  if (!counts[1]) {
    if (labels) {
      const int32_t lab = labels[i];
      keep = lab >= 0 && sizes[lab] >= min_size;
    } else {
      keep = w.parent[i] != kCompNone;
    }
  }
  w.g.avg[i] = keep ? 1.0 : 0.0;
}

// grid, boxes and counts: the part both entries share
static int cl_prepare(const ClusterWs &w, const float *d_xyz, const uint32_t *d_count, const float *d_bounds, double eps,
                      uint32_t thr, uint32_t *d_out_counts, cudaStream_t st) {
  const uint32_t n = w.cap_rows;
  const uint32_t blocks = (n + kClThreads - 1) / kClThreads;
  const double eps2 = eps * eps;
  if (cudaMemsetAsync(d_out_counts, 0, 4 * sizeof(uint32_t), st) != cudaSuccess ||
      cudaMemsetAsync(w.box, 0xFF, (size_t)n * 12, st) != cudaSuccess ||
      cudaMemsetAsync(w.box + 3 * (size_t)n, 0, (size_t)n * 12, st) != cudaSuccess ||
      cudaMemsetAsync(w.rep, 0xFF, (size_t)n * 4, st) != cudaSuccess)
    return record_cuda_error(cudaGetLastError());
  const int rc = sor_grid_build_fixed(w.g, d_xyz, d_count, d_bounds, eps * 0.5 * (1.0 + 0x1p-20), n, d_out_counts + 1, st);
  if (rc != D2PC_OK) return rc;
  cl_box_kernel<<<blocks, kClThreads, 0, st>>>(w, d_out_counts);
  D2PC_CHECK_LAUNCH();
  cl_count_kernel<<<blocks, kClThreads, 0, st>>>(w, eps2, thr, d_out_counts);
  D2PC_CHECK_LAUNCH();
  return D2PC_OK;
}

static bool cl_eps_ok(double eps) {
  return eps > 0.0 && eps * eps > 0.0 && eps * eps < __builtin_huge_val();
}

}  // namespace d2pc

using namespace d2pc;

extern "C" int d2pc_cluster_scratch_bytes(uint32_t capacity_rows, size_t *bytes) {
  if (!bytes || capacity_rows == 0) return D2PC_ERR_INVALID_ARGUMENT;
  *bytes = cluster_ws_bytes(capacity_rows);
  return D2PC_OK;
}

extern "C" int d2pc_radius_outlier_enqueue(const float *d_xyz, const float *d_rgb, const uint32_t *d_count,
                                           uint32_t capacity_rows, const float *d_bounds, int32_t nb_points,
                                           double radius, void *d_scratch, size_t scratch_bytes, float *d_out_xyz,
                                           float *d_out_rgb, uint32_t *d_out_index, uint32_t *d_out_counts,
                                           void *stream) {
  if (!d_xyz || !d_count || !d_bounds || !d_scratch || !d_out_xyz || !d_out_counts) return D2PC_ERR_INVALID_ARGUMENT;
  if ((d_out_rgb != nullptr) != (d_rgb != nullptr)) return D2PC_ERR_INVALID_ARGUMENT;
  if (capacity_rows == 0 || nb_points < 1 || !cl_eps_ok(radius)) return D2PC_ERR_INVALID_ARGUMENT;
  if (((uintptr_t)d_scratch & 255u) != 0) return D2PC_ERR_INVALID_ARGUMENT;
  if (scratch_bytes < cluster_ws_bytes(capacity_rows)) return D2PC_ERR_WORKSPACE_TOO_SMALL;
  cudaStream_t st = (cudaStream_t)stream;
  const ClusterWs w = cluster_ws(d_scratch, capacity_rows);
  const uint32_t blocks = (capacity_rows + kClThreads - 1) / kClThreads;
  int rc = cl_prepare(w, d_xyz, d_count, d_bounds, radius, (uint32_t)nb_points + 1u, d_out_counts, st);
  if (rc != D2PC_OK) return rc;
  cl_keep_kernel<<<blocks, kClThreads, 0, st>>>(w, nullptr, nullptr, 0u, d_out_counts);
  D2PC_CHECK_LAUNCH();
  return sor_compact(w.g, d_xyz, d_rgb, d_out_xyz, d_out_rgb, d_out_index, d_out_counts, capacity_rows, st);
}

extern "C" int d2pc_dbscan_enqueue(const float *d_xyz, const float *d_rgb, const uint32_t *d_count,
                                   uint32_t capacity_rows, const float *d_bounds, double eps, int32_t min_points,
                                   uint32_t min_size, void *d_scratch, size_t scratch_bytes, int32_t *d_out_labels,
                                   uint32_t *d_out_sizes, float *d_out_xyz, float *d_out_rgb, uint32_t *d_out_index,
                                   uint32_t *d_out_counts, void *stream) {
  if (!d_xyz || !d_count || !d_bounds || !d_scratch || !d_out_labels || !d_out_sizes || !d_out_counts)
    return D2PC_ERR_INVALID_ARGUMENT;
  if ((d_out_rgb != nullptr) != (d_rgb != nullptr && d_out_xyz != nullptr)) return D2PC_ERR_INVALID_ARGUMENT;
  if (!d_out_xyz && d_out_index) return D2PC_ERR_INVALID_ARGUMENT;
  if (capacity_rows == 0 || min_points < 0 || min_size < 1 || !cl_eps_ok(eps)) return D2PC_ERR_INVALID_ARGUMENT;
  if (((uintptr_t)d_scratch & 255u) != 0) return D2PC_ERR_INVALID_ARGUMENT;
  if (scratch_bytes < cluster_ws_bytes(capacity_rows)) return D2PC_ERR_WORKSPACE_TOO_SMALL;
  cudaStream_t st = (cudaStream_t)stream;
  const ClusterWs w = cluster_ws(d_scratch, capacity_rows);
  const uint32_t blocks = (capacity_rows + kClThreads - 1) / kClThreads;
  const double eps2 = eps * eps;
  if (cudaMemsetAsync(d_out_sizes, 0, (size_t)capacity_rows * 4, st) != cudaSuccess)
    return record_cuda_error(cudaGetLastError());
  int rc = cl_prepare(w, d_xyz, d_count, d_bounds, eps, min_points > 1 ? (uint32_t)min_points : 1u, d_out_counts, st);
  if (rc != D2PC_OK) return rc;
  cl_rep_kernel<<<blocks, kClThreads, 0, st>>>(w, d_out_counts);
  D2PC_CHECK_LAUNCH();
  cl_unite_cell_kernel<<<blocks, kClThreads, 0, st>>>(w, d_out_counts);
  D2PC_CHECK_LAUNCH();
  cl_unite_near_kernel<<<blocks, kClThreads, 0, st>>>(w, eps2, d_out_counts);
  D2PC_CHECK_LAUNCH();
  cl_root_count_kernel<<<blocks, kClThreads, 0, st>>>(w, d_out_counts);
  D2PC_CHECK_LAUNCH();
  tile_scan_kernel<<<1, kTileScanThreads, 0, st>>>(w.g.tile_cnt, blocks, d_out_counts + 2);
  D2PC_CHECK_LAUNCH();
  cl_root_id_kernel<<<blocks, kClThreads, 0, st>>>(w, d_out_counts);
  D2PC_CHECK_LAUNCH();
  cl_core_label_kernel<<<blocks, kClThreads, 0, st>>>(w, d_out_labels, d_out_counts);
  D2PC_CHECK_LAUNCH();
  cl_border_kernel<<<blocks, kClThreads, 0, st>>>(w, eps2, d_out_labels, d_out_counts);
  D2PC_CHECK_LAUNCH();
  cl_sizes_kernel<<<blocks, kClThreads, 0, st>>>(w, d_out_labels, d_out_sizes, d_out_counts);
  D2PC_CHECK_LAUNCH();
  if (!d_out_xyz) return D2PC_OK;
  cl_keep_kernel<<<blocks, kClThreads, 0, st>>>(w, d_out_labels, d_out_sizes, min_size, d_out_counts);
  D2PC_CHECK_LAUNCH();
  return sor_compact(w.g, d_xyz, d_rgb, d_out_xyz, d_out_rgb, d_out_index, d_out_counts, capacity_rows, st);
}
