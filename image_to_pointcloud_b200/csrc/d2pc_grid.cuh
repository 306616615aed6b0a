// d2pc_grid.cuh -- the hashed uniform grid behind the exact k-nearest-neighbour searches (statistical outlier
// removal in d2pc_sor.cu, normals in d2pc_normals.cu): header and workspace layout, the cell hash table, cell
// coordinates, and the host sequence that builds the grid (sor_grid_build, defined in d2pc_sor.cu next to its
// kernels).  After the build, `sorted` / `sorted_idx` hold the points in slot order, `cell_off` the first sorted
// point of every slot, heavy cells are sorted by x and flagged in `cell_cnt`.
#ifndef D2PC_GRID_CUH_
#define D2PC_GRID_CUH_

#include "d2pc_device.cuh"

namespace d2pc {

constexpr int kSorMaxK = 64;
constexpr int kSorThreads = 256;
constexpr int kSorScanThreads = 1024;
constexpr int kSorTrials = 8;
constexpr double kSorTrialStep = 1.5;     // ratio between consecutive candidate cell sizes
constexpr double kSorTargetOcc = 5.0;     // points per occupied cell aimed at
constexpr int kSorCoordBits = 20;         // cell coordinates per axis
constexpr unsigned long long kSorEmpty = 0xFFFFFFFFFFFFFFFFull;
// Very heavy cells.  Every cloud of this stage contains a structure far smaller than any sensible cell: the
// pixels clipped at a percentile all get the same tiny z and collapse into a lattice ~1e-7 wide (2% of the
// points: 42 000 at 1080p, 166 000 at 4K).  They share one cell, and comparing them pairwise is quadratic.
// Cells above kSorHeavyMin points are therefore sorted by x (one CTA per cell), and a query walks only the
// window |dx| <= its current k-th distance, outwards from its own x.
constexpr uint32_t kSorHeavyMin = 4096;
constexpr uint32_t kSorHeavyMax = 1u << 20;    // one CTA sorts one cell (bitonic, L2 resident)
constexpr uint32_t kSorMaxHeavy = 256;         // heavy cells handled per call (the rest stay plain lists)
constexpr uint32_t kSorSortedFlag = 0x80000000u;

struct __align__(256) SorHeader {
  double mn[3], ext[3];
  double h, slack;
  double trial_h[kSorTrials];
  uint32_t trial_occ[kSorTrials];
  int32_t dim[3];       // cells per axis for the chosen size (coordinates are clamped to it)
  uint32_t n, chosen;
  double cloud_mean, std_dev, thr;
  uint32_t n_heavy, heavy_total;
};

struct SorWs {
  SorHeader *hdr;
  unsigned long long *keys;  // [cap]     cell key per table slot (kSorEmpty = free)
  uint32_t *cell_off;        // [cap + 1] first sorted point of every slot
  uint32_t *cell_cnt;        // [cap]     counts, then scatter cursors
  uint32_t *blk_sum;         // [cap / 1024 + 1] (>= 256 doubles: reused by the statistics)
  uint32_t *pt_cell;         // [N]       slot of every point
  float *sorted;             // [N][3]    points in slot order
  uint32_t *sorted_idx;      // [N]       source row of every sorted point
  double *avg;               // [N]
  uint32_t *tile_cnt;        // [N / 256 + 1]
  uint32_t *heavy;           // [2 * kSorMaxHeavy] slot, offset into `pairs`
  unsigned long long *pairs; // [2 N] (x key << 32 | rank) per heavy cell, padded to a power of two
  float *tmp_xyz;            // [N][3] scratch for the permutation
  uint32_t *tmp_idx;         // [N]
  uint32_t cap;              // table slots: power of two >= 2 N
};

inline uint32_t sor_capacity(uint32_t n_rows) {
  uint32_t c = 1u << 16;
  while (c < 2u * n_rows && c < 0x80000000u) c <<= 1;
  return c;
}
inline size_t sor_ws_bytes(uint32_t n_rows) {
  const size_t cap = sor_capacity(n_rows);
  size_t b = sizeof(SorHeader);
  b += align_up(cap * 8, 256) + align_up((cap + 1) * 4, 256) + align_up(cap * 4, 256);
  b += align_up((cap / kSorScanThreads + 1) * 4 + 2048, 256);   // + room for 256 float64 partial sums
  b += 2 * align_up((size_t)n_rows * 4, 256) + align_up((size_t)n_rows * 12, 256) + align_up((size_t)n_rows * 8, 256);
  b += align_up((size_t)(n_rows / kSorThreads + 1) * 4, 256);
  b += align_up((size_t)2 * kSorMaxHeavy * 4, 256) + align_up((size_t)2 * n_rows * 8 + 8, 256);
  b += align_up((size_t)n_rows * 12, 256) + align_up((size_t)n_rows * 4, 256);
  return b;
}
inline SorWs sor_ws(void *base, uint32_t n_rows) {
  SorWs w;
  const size_t cap = sor_capacity(n_rows);
  char *p = (char *)base;
  w.hdr = (SorHeader *)p;               p += sizeof(SorHeader);
  w.keys = (unsigned long long *)p;     p += align_up(cap * 8, 256);
  w.cell_off = (uint32_t *)p;           p += align_up((cap + 1) * 4, 256);
  w.cell_cnt = (uint32_t *)p;           p += align_up(cap * 4, 256);
  w.blk_sum = (uint32_t *)p;            p += align_up((cap / kSorScanThreads + 1) * 4 + 2048, 256);
  w.pt_cell = (uint32_t *)p;            p += align_up((size_t)n_rows * 4, 256);
  w.sorted = (float *)p;                p += align_up((size_t)n_rows * 12, 256);
  w.sorted_idx = (uint32_t *)p;         p += align_up((size_t)n_rows * 4, 256);
  w.avg = (double *)p;                  p += align_up((size_t)n_rows * 8, 256);
  w.tile_cnt = (uint32_t *)p;           p += align_up((size_t)(n_rows / kSorThreads + 1) * 4, 256);
  w.heavy = (uint32_t *)p;              p += align_up((size_t)2 * kSorMaxHeavy * 4, 256);
  w.pairs = (unsigned long long *)p;    p += align_up((size_t)2 * n_rows * 8 + 8, 256);
  w.tmp_xyz = (float *)p;               p += align_up((size_t)n_rows * 12, 256);
  w.tmp_idx = (uint32_t *)p;
  w.cap = (uint32_t)cap;
  return w;
}

// Enqueues the grid build on `st` (begin, cell-size trials, choose, count, scan, scatter, heavy cells): every
// launch from sor_begin_kernel to sor_heavy_sort_kernel.  Returns D2PC_OK or the launch error.
int sor_grid_build(const SorWs &w, const float *d_xyz, const uint32_t *d_count, const float *d_bounds,
                   uint32_t capacity_rows, cudaStream_t st);

// The same grid with the cell size `cs` given (begin, clear, count, scan, scatter; no heavy cells).  *d_err gets
// D2PC_CLUSTER_ERR_GRID when an axis of the box would need kSorCellLimit cells or more, else 0.
constexpr double kSorCellLimit = 1048574.0;   // cells per axis below which sor_cell_coords never clamps
int sor_grid_build_fixed(const SorWs &w, const float *d_xyz, const uint32_t *d_count, const float *d_bounds, double cs,
                         uint32_t capacity_rows, uint32_t *d_err, cudaStream_t st);

// Ordered compaction of the rows with 0 < avg[i] < hdr->thr (keep counts per tile, scan, copy) into d_out_* with
// their source rows; *d_out_count = kept rows.
int sor_compact(const SorWs &w, const float *d_xyz, const float *d_rgb, float *d_out_xyz, float *d_out_rgb,
                uint32_t *d_out_index, uint32_t *d_out_count, uint32_t capacity_rows, cudaStream_t st);

#if defined(__CUDACC__)
__device__ __forceinline__ uint32_t sor_hash(unsigned long long k) {
  k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
  return (uint32_t)k;
}
__device__ __forceinline__ unsigned long long sor_key(int32_t c0, int32_t c1, int32_t c2) {
  return ((unsigned long long)(uint32_t)c0 << (2 * kSorCoordBits)) | ((unsigned long long)(uint32_t)c1 << kSorCoordBits) |
         (unsigned long long)(uint32_t)c2;
}

__device__ __forceinline__ void sor_cell_coords(const SorHeader *h, double cs, double x, double y, double z, int32_t c[3]) {
  const double p[3] = {x, y, z};
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    double q = floor((p[a] - h->mn[a]) / cs);
    const double top = floor(h->ext[a] / cs);  // last cell of the axis: the maximum itself must not open a new one
    q = q < top ? q : top;
    c[a] = q > 0.0 ? (q < 1048574.0 ? (int32_t)q : 1048574) : 0;  // NaN -> 0
  }
}

// insert a key; returns the slot, *fresh = this call created the entry
__device__ __forceinline__ uint32_t sor_insert(const SorWs &w, unsigned long long key, bool *fresh) {
  const uint32_t mask = w.cap - 1u;
  uint32_t slot = sor_hash(key) & mask;
  *fresh = false;
  while (true) {
    unsigned long long k = *reinterpret_cast<volatile unsigned long long *>(&w.keys[slot]);
    if (k == kSorEmpty) {
      k = atomicCAS(&w.keys[slot], kSorEmpty, key);
      if (k == kSorEmpty) { *fresh = true; return slot; }
    }
    if (k == key) return slot;
    slot = (slot + 1u) & mask;
  }
}
__device__ __forceinline__ bool sor_find(const SorWs &w, unsigned long long key, uint32_t *slot_out) {
  const uint32_t mask = w.cap - 1u;
  uint32_t slot = sor_hash(key) & mask;
  while (true) {
    const unsigned long long k = w.keys[slot];
    if (k == key) { *slot_out = slot; return true; }
    if (k == kSorEmpty) return false;
    slot = (slot + 1u) & mask;
  }
}

// float32 upper bound of the current k-th squared distance (inf while fewer than k points were seen)
__device__ __forceinline__ float sor_filter(double kth) {
  return __double2float_ru(kth) * 1.000001f;
}
#endif  // __CUDACC__

}  // namespace d2pc
#endif  // D2PC_GRID_CUH_
