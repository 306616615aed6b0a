// d2pc_serialise.cu -- row f3: the byte layouts the reference's writers and preview produce
// (backend/app.py:310-389, 495-506), generated on the device from the emitted rows so that only
// the bytes a file or the preview JSON needs cross PCIe and no per-point host loop remains
// (save_xyz is a Python loop over every point in the reference, app.py:383-387).
//   preview rows   points[::stride], colors[::stride]                       -> d2pc_preview_rows_enqueue
//   XYZ ASCII      "%.6f %.6f %.6f %d %d %d\n" per row, variable length       -> d2pc_xyz_text_*_enqueue
//                  (measure: per-tile byte counts + scan; write: format into shared memory at
//                  the row's offset, 16-byte coalesced copy-out)
//   LAS 1.2 fmt 2  26-byte records, scaled int32 coordinates, 16-bit colours  -> d2pc_las_records_enqueue
//   PLY (Open3D)   27-byte records, float64 coordinates, uchar colours        -> d2pc_ply_records_enqueue
//                  51-byte records, + float64 normals                        -> d2pc_ply_normal_records_enqueue
//                  13-byte mesh faces, uchar 3 + three uint32 vertex ids     -> d2pc_ply_face_records_enqueue
// Every entry point works on ONE frame's rows (pointers into the [batch, N, 3] outputs of emit).
#include "d2pc_device.cuh"
#include "d2pc_format.h"

namespace d2pc {

constexpr int kSerThreads = 256;           // rows per CTA (one row per thread)
constexpr uint32_t kSerMaxRows = 1u << 24;  // keeps every byte offset below 2^32

__global__ void __launch_bounds__(kSerThreads) ser_preview_kernel(const float *xyz, const float *rgb, const uint32_t *count,
                                                                  uint32_t max_preview, float *oxyz, float *orgb,
                                                                  uint32_t out_cap, uint32_t *ocount) {
  const uint32_t n = *count;
  const uint32_t stride = preview_stride(n, max_preview);
  const uint32_t rows = n == 0u ? 0u : (n - 1u) / stride + 1u;  // len(points[::stride])
  const uint32_t m = min(rows, out_cap);
  if (blockIdx.x == 0 && threadIdx.x == 0) *ocount = m;
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < m; j += gridDim.x * blockDim.x) {
    const size_t src = 3 * (size_t)j * stride, dst = 3 * (size_t)j;
#pragma unroll
    for (int k = 0; k < 3; ++k) { oxyz[dst + k] = __ldg(xyz + src + k); orgb[dst + k] = __ldg(rgb + src + k); }
  }
}

// ---- XYZ ASCII -------------------------------------------------------------------------------
__global__ void __launch_bounds__(kSerThreads) ser_xyz_len_kernel(const float *xyz, const float *rgb, const uint32_t *count,
                                                                  uint32_t *tile_bytes, int32_t *err) {
  __shared__ uint32_t s_warp[kSerThreads / 32];
  const uint32_t n = *count;
  const uint32_t i = blockIdx.x * (uint32_t)kSerThreads + threadIdx.x;
  uint32_t len = 0;
  if (i < n) {
    char line[kXyzMaxLine];
    float p[3], c[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) { p[k] = __ldg(xyz + 3 * (size_t)i + k); c[k] = __ldg(rgb + 3 * (size_t)i + k); }
    const int m = format_xyz_line(p, c, line);
    if (m < 0) *err = 1; else len = (uint32_t)m;
  }
  len = warp_sum(len);
  if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = len;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t t = 0;
    for (int w = 0; w < kSerThreads / 32; ++w) t += s_warp[w];
    tile_bytes[blockIdx.x] = t;
  }
}

// exclusive scan of the per-tile byte counts (in place), total -> *total_bytes
__global__ void __launch_bounds__(1024) ser_scan_kernel(uint32_t *tile_bytes, uint32_t n_tiles, unsigned long long *total_bytes) {
  __shared__ uint32_t s_warp[32];
  __shared__ uint32_t s_carry;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_carry = 0;
  __syncthreads();
  for (uint32_t base = 0; base < n_tiles; base += 1024u) {
    const uint32_t i = base + (uint32_t)tid;
    const uint32_t c = i < n_tiles ? tile_bytes[i] : 0u;
    uint32_t incl = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t y = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += y;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    uint32_t woff = 0, total = 0;
    for (int w = 0; w < 32; ++w) { const uint32_t x = s_warp[w]; if (w < warp) woff += x; total += x; }
    if (i < n_tiles) tile_bytes[i] = s_carry + woff + incl - c;
    __syncthreads();
    if (tid == 0) s_carry += total;
    __syncthreads();
  }
  if (tid == 0) *total_bytes = (unsigned long long)s_carry;
}

// 16-byte coalesced copy of n bytes from shared staging to global; staging byte s_off corresponds
// to global byte g0 (s_off == g0 & 15, so source and destination share alignment)
__device__ __forceinline__ void copy_bytes_out(const uint8_t *s, uint32_t s_off, uint32_t n, uint8_t *gbase, size_t g0) {
  uint8_t *galigned = gbase + (g0 - s_off);
  const uint32_t span = s_off + n;
  const uint32_t chunks = (span + 15u) >> 4;
  for (uint32_t c = threadIdx.x; c < chunks; c += blockDim.x) {
    const uint32_t w = c << 4;
    if (w >= s_off && w + 16u <= span) {
      *reinterpret_cast<uint4 *>(galigned + w) = *reinterpret_cast<const uint4 *>(s + w);
    } else {
      for (uint32_t k = 0; k < 16u; ++k)
        if (w + k >= s_off && w + k < span) galigned[w + k] = s[w + k];
    }
  }
}

__global__ void __launch_bounds__(kSerThreads) ser_xyz_write_kernel(const float *xyz, const float *rgb, const uint32_t *count,
                                                                    const uint32_t *tile_off, char *text,
                                                                    unsigned long long text_cap,
                                                                    const unsigned long long *total_bytes,
                                                                    const int32_t *err) {
  __shared__ __align__(16) uint8_t s_text[kSerThreads * kXyzMaxLine + 16];
  __shared__ uint32_t s_warp[kSerThreads / 32];
  const uint32_t n = *count;
  const uint32_t tile_base = blockIdx.x * (uint32_t)kSerThreads;
  if (tile_base >= n || *err != 0 || *total_bytes > text_cap) return;  // uniform
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t i = tile_base + threadIdx.x;
  char line[kXyzMaxLine];
  uint32_t len = 0;
  if (i < n) {
    float p[3], c[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) { p[k] = __ldg(xyz + 3 * (size_t)i + k); c[k] = __ldg(rgb + 3 * (size_t)i + k); }
    const int m = format_xyz_line(p, c, line);
    len = m < 0 ? 0u : (uint32_t)m;
  }
  uint32_t incl = len;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t y = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += y;
  }
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();
  uint32_t woff = 0, total = 0;
#pragma unroll
  for (int w = 0; w < kSerThreads / 32; ++w) { const uint32_t x = s_warp[w]; if (w < warp) woff += x; total += x; }
  const size_t g0 = (size_t)tile_off[blockIdx.x];
  const uint32_t s_off = (uint32_t)(((uintptr_t)text + g0) & 15u);
  uint8_t *dst = s_text + s_off + woff + incl - len;
  for (uint32_t k = 0; k < len; ++k) dst[k] = (uint8_t)line[k];
  __syncthreads();
  copy_bytes_out(s_text, s_off, total, reinterpret_cast<uint8_t *>(text), g0);
}

// ---- fixed-size records (LAS 26 B, PLY 27 B): staged per CTA, written as 16-byte words ---------
template <int REC, typename F>
__device__ __forceinline__ void ser_records(const uint32_t *count, uint8_t *records, F make) {
  __shared__ __align__(16) uint8_t s_rec[kSerThreads * REC];
  const uint32_t n = *count;
  const uint32_t tile_base = blockIdx.x * (uint32_t)kSerThreads;
  if (tile_base >= n) return;
  const uint32_t i = tile_base + threadIdx.x;
  if (i < n) make(i, s_rec + (size_t)threadIdx.x * REC);
  __syncthreads();
  const uint32_t rows = min((uint32_t)kSerThreads, n - tile_base);
  const size_t g0 = (size_t)tile_base * REC;  // 256 * REC is a multiple of 16
  copy_bytes_out(s_rec, 0u, rows * REC, records, g0);  // records is 16 B-aligned (checked by the host)
}

__global__ void __launch_bounds__(kSerThreads) ser_las_kernel(const float *xyz, const float *rgb, const uint32_t *count,
                                                              const float *bounds, double scale, uint8_t *records,
                                                              int32_t *int_minmax, int32_t *err) {
  __shared__ int32_t s_mm[6];
  if (threadIdx.x < 6) s_mm[threadIdx.x] = threadIdx.x < 3 ? 2147483647 : (-2147483647 - 1);
  __syncthreads();
  const double off[3] = {(double)bounds[0], (double)bounds[1], (double)bounds[2]};  // float(points[:, k].min())
  ser_records<kLasRecordBytes>(count, records, [&](uint32_t i, uint8_t *o) {
    float p[3], c[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) { p[k] = __ldg(xyz + 3 * (size_t)i + k); c[k] = __ldg(rgb + 3 * (size_t)i + k); }
    int32_t q[3];
    if (!las_record(p, c, off, scale, o, q)) *err = 1;
#pragma unroll
    for (int k = 0; k < 3; ++k) { atomicMin(&s_mm[k], q[k]); atomicMax(&s_mm[3 + k], q[k]); }
  });
  __syncthreads();
  if (threadIdx.x < 6 && blockIdx.x * (uint32_t)kSerThreads < *count) {
    if (threadIdx.x < 3) atomicMin(&int_minmax[threadIdx.x], s_mm[threadIdx.x]);
    else atomicMax(&int_minmax[threadIdx.x], s_mm[threadIdx.x]);
  }
}

__global__ void __launch_bounds__(kSerThreads) ser_ply_kernel(const float *xyz, const float *rgb, const uint32_t *count,
                                                              uint8_t *records) {
  ser_records<kPlyRecordBytes>(count, records, [&](uint32_t i, uint8_t *o) {
    float p[3], c[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) { p[k] = __ldg(xyz + 3 * (size_t)i + k); c[k] = __ldg(rgb + 3 * (size_t)i + k); }
    ply_record(p, c, o);
  });
}

__global__ void __launch_bounds__(kSerThreads) ser_ply_normal_kernel(const float *xyz, const double *normals,
                                                                     const float *rgb, const uint32_t *count,
                                                                     uint8_t *records) {
  ser_records<kPlyNormalRecordBytes>(count, records, [&](uint32_t i, uint8_t *o) {
    float p[3], c[3];
    double nv[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      p[k] = __ldg(xyz + 3 * (size_t)i + k);
      nv[k] = __ldg(normals + 3 * (size_t)i + k);
      c[k] = __ldg(rgb + 3 * (size_t)i + k);
    }
    ply_normal_record(p, nv, c, o);
  });
}

__global__ void __launch_bounds__(kSerThreads) ser_ply_face_kernel(const int32_t *tri, const uint32_t *count,
                                                                   uint8_t *records) {
  ser_records<kPlyFaceRecordBytes>(count, records, [&](uint32_t i, uint8_t *o) {
    int32_t t[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) t[k] = __ldg(tri + 3 * (size_t)i + k);
    ply_face_record(t, o);
  });
}

// per-axis min / max of the rows (float(points[:, k].min()), app.py:352, 394-399) when emit's fused bounds
// are not at hand: keys[0..2] = min, keys[3..5] = max (ordered uint32 keys)
__global__ void ser_bounds_init_kernel(uint32_t *keys) {
  if (threadIdx.x < 6) keys[threadIdx.x] = threadIdx.x < 3 ? 0xFFFFFFFFu : 0u;
}
__global__ void __launch_bounds__(kSerThreads) ser_bounds_kernel(const float *xyz, const uint32_t *count, uint32_t *keys) {
  __shared__ uint32_t s_k[6];
  if (threadIdx.x < 6) s_k[threadIdx.x] = threadIdx.x < 3 ? 0xFFFFFFFFu : 0u;
  __syncthreads();
  const uint32_t n = *count;
  uint32_t lo[3] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu}, hi[3] = {0u, 0u, 0u};
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const float v = __ldg(xyz + 3 * (size_t)i + k);
      if (v == v) {  // NaN would poison numpy's min / max; callers never pass it
        const uint32_t key = float_to_key(v);
        lo[k] = min(lo[k], key);
        hi[k] = max(hi[k], key);
      }
    }
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const uint32_t a = warp_min(lo[k]), b = warp_max(hi[k]);
    if ((threadIdx.x & 31) == 0) { atomicMin(&s_k[k], a); atomicMax(&s_k[3 + k], b); }
  }
  __syncthreads();
  if (threadIdx.x < 3) atomicMin(&keys[threadIdx.x], s_k[threadIdx.x]);
  else if (threadIdx.x < 6) atomicMax(&keys[threadIdx.x], s_k[threadIdx.x]);
}
__global__ void ser_bounds_export_kernel(const uint32_t *keys, float *out) {
  if (threadIdx.x < 6) {
    const bool empty = keys[0] == 0xFFFFFFFFu && keys[3] == 0u;
    out[threadIdx.x] = empty ? nan_f32() : key_to_float(keys[threadIdx.x]);
  }
}

__global__ void ser_las_init_kernel(int32_t *int_minmax, int32_t *err) {
  if (threadIdx.x < 6) int_minmax[threadIdx.x] = threadIdx.x < 3 ? 2147483647 : (-2147483647 - 1);
  if (threadIdx.x == 0) *err = 0;
}

}  // namespace d2pc

using namespace d2pc;

static inline uint32_t ser_tiles(uint32_t rows) { return (rows + kSerThreads - 1) / kSerThreads; }

extern "C" int d2pc_preview_rows_enqueue(const float *d_xyz, const float *d_rgb, const uint32_t *d_count,
                                         uint32_t max_preview, float *d_out_xyz, float *d_out_rgb,
                                         uint32_t out_capacity_rows, uint32_t *d_out_count, void *stream) {
  if (!d_xyz || !d_rgb || !d_count || !d_out_xyz || !d_out_rgb || !d_out_count) return D2PC_ERR_INVALID_ARGUMENT;
  const uint32_t blocks = out_capacity_rows == 0 ? 1u : min(ser_tiles(out_capacity_rows), 148u * 8u);
  ser_preview_kernel<<<blocks, kSerThreads, 0, (cudaStream_t)stream>>>(d_xyz, d_rgb, d_count, max_preview, d_out_xyz,
                                                                      d_out_rgb, out_capacity_rows, d_out_count);
  D2PC_CHECK_LAUNCH();
  return D2PC_OK;
}

extern "C" int d2pc_xyz_text_scratch_bytes(uint32_t capacity_rows, size_t *bytes) {
  if (!bytes || capacity_rows == 0 || capacity_rows >= kSerMaxRows) return D2PC_ERR_INVALID_ARGUMENT;
  *bytes = align_up((size_t)ser_tiles(capacity_rows) * sizeof(uint32_t), 256);
  return D2PC_OK;
}

extern "C" int d2pc_xyz_text_measure_enqueue(const float *d_xyz, const float *d_rgb, const uint32_t *d_count,
                                             uint32_t capacity_rows, void *d_scratch, size_t scratch_bytes,
                                             unsigned long long *d_text_bytes, int32_t *d_error, void *stream) {
  if (!d_xyz || !d_rgb || !d_count || !d_scratch || !d_text_bytes || !d_error) return D2PC_ERR_INVALID_ARGUMENT;
  if (capacity_rows == 0 || capacity_rows >= kSerMaxRows) return D2PC_ERR_INVALID_ARGUMENT;
  const uint32_t tiles = ser_tiles(capacity_rows);
  if (scratch_bytes < (size_t)tiles * sizeof(uint32_t)) return D2PC_ERR_WORKSPACE_TOO_SMALL;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(d_error, 0, sizeof(int32_t), st);
  if (e != cudaSuccess) return record_cuda_error(e);
  ser_xyz_len_kernel<<<tiles, kSerThreads, 0, st>>>(d_xyz, d_rgb, d_count, (uint32_t *)d_scratch, d_error);
  D2PC_CHECK_LAUNCH();
  ser_scan_kernel<<<1, 1024, 0, st>>>((uint32_t *)d_scratch, tiles, d_text_bytes);
  D2PC_CHECK_LAUNCH();
  return D2PC_OK;
}

extern "C" int d2pc_xyz_text_write_enqueue(const float *d_xyz, const float *d_rgb, const uint32_t *d_count,
                                           uint32_t capacity_rows, const void *d_scratch, size_t scratch_bytes,
                                           const unsigned long long *d_text_bytes, const int32_t *d_error, char *d_text,
                                           size_t text_capacity, void *stream) {
  if (!d_xyz || !d_rgb || !d_count || !d_scratch || !d_text_bytes || !d_error || !d_text) return D2PC_ERR_INVALID_ARGUMENT;
  if (capacity_rows == 0 || capacity_rows >= kSerMaxRows) return D2PC_ERR_INVALID_ARGUMENT;
  const uint32_t tiles = ser_tiles(capacity_rows);
  if (scratch_bytes < (size_t)tiles * sizeof(uint32_t)) return D2PC_ERR_WORKSPACE_TOO_SMALL;
  ser_xyz_write_kernel<<<tiles, kSerThreads, 0, (cudaStream_t)stream>>>(d_xyz, d_rgb, d_count, (const uint32_t *)d_scratch,
                                                                       d_text, (unsigned long long)text_capacity,
                                                                       d_text_bytes, d_error);
  D2PC_CHECK_LAUNCH();
  return D2PC_OK;
}

extern "C" int d2pc_rows_bounds_enqueue(const float *d_xyz, const uint32_t *d_count, uint32_t capacity_rows,
                                        uint32_t *d_scratch6, float *d_bounds6, void *stream) {
  if (!d_xyz || !d_count || !d_scratch6 || !d_bounds6 || capacity_rows == 0) return D2PC_ERR_INVALID_ARGUMENT;
  cudaStream_t st = (cudaStream_t)stream;
  ser_bounds_init_kernel<<<1, 32, 0, st>>>(d_scratch6);
  D2PC_CHECK_LAUNCH();
  ser_bounds_kernel<<<min(ser_tiles(capacity_rows), 148u * 8u), kSerThreads, 0, st>>>(d_xyz, d_count, d_scratch6);
  D2PC_CHECK_LAUNCH();
  ser_bounds_export_kernel<<<1, 32, 0, st>>>(d_scratch6, d_bounds6);
  D2PC_CHECK_LAUNCH();
  return D2PC_OK;
}

extern "C" int d2pc_las_records_enqueue(const float *d_xyz, const float *d_rgb, const uint32_t *d_count,
                                        uint32_t capacity_rows, const float *d_bounds, double scale, uint8_t *d_records,
                                        int32_t *d_int_minmax, int32_t *d_error, void *stream) {
  if (!d_xyz || !d_rgb || !d_count || !d_bounds || !d_records || !d_int_minmax || !d_error) return D2PC_ERR_INVALID_ARGUMENT;
  if (capacity_rows == 0 || !(scale > 0.0) || ((uintptr_t)d_records & 15u) != 0) return D2PC_ERR_INVALID_ARGUMENT;
  cudaStream_t st = (cudaStream_t)stream;
  ser_las_init_kernel<<<1, 32, 0, st>>>(d_int_minmax, d_error);
  D2PC_CHECK_LAUNCH();
  ser_las_kernel<<<ser_tiles(capacity_rows), kSerThreads, 0, st>>>(d_xyz, d_rgb, d_count, d_bounds, scale, d_records,
                                                                   d_int_minmax, d_error);
  D2PC_CHECK_LAUNCH();
  return D2PC_OK;
}

extern "C" int d2pc_ply_records_enqueue(const float *d_xyz, const float *d_rgb, const uint32_t *d_count,
                                        uint32_t capacity_rows, uint8_t *d_records, void *stream) {
  if (!d_xyz || !d_rgb || !d_count || !d_records) return D2PC_ERR_INVALID_ARGUMENT;
  if (capacity_rows == 0 || ((uintptr_t)d_records & 15u) != 0) return D2PC_ERR_INVALID_ARGUMENT;
  ser_ply_kernel<<<ser_tiles(capacity_rows), kSerThreads, 0, (cudaStream_t)stream>>>(d_xyz, d_rgb, d_count, d_records);
  D2PC_CHECK_LAUNCH();
  return D2PC_OK;
}

extern "C" int d2pc_ply_normal_records_enqueue(const float *d_xyz, const double *d_normals, const float *d_rgb,
                                               const uint32_t *d_count, uint32_t capacity_rows, uint8_t *d_records,
                                               void *stream) {
  if (!d_xyz || !d_normals || !d_rgb || !d_count || !d_records) return D2PC_ERR_INVALID_ARGUMENT;
  if (capacity_rows == 0 || ((uintptr_t)d_records & 15u) != 0) return D2PC_ERR_INVALID_ARGUMENT;
  ser_ply_normal_kernel<<<ser_tiles(capacity_rows), kSerThreads, 0, (cudaStream_t)stream>>>(d_xyz, d_normals, d_rgb,
                                                                                            d_count, d_records);
  D2PC_CHECK_LAUNCH();
  return D2PC_OK;
}

extern "C" int d2pc_ply_face_records_enqueue(const int32_t *d_tri, const uint32_t *d_tri_count, uint32_t capacity,
                                             uint8_t *d_records, void *stream) {
  if (!d_tri || !d_tri_count || !d_records) return D2PC_ERR_INVALID_ARGUMENT;
  if (capacity == 0 || ((uintptr_t)d_records & 15u) != 0) return D2PC_ERR_INVALID_ARGUMENT;
  ser_ply_face_kernel<<<ser_tiles(capacity), kSerThreads, 0, (cudaStream_t)stream>>>(d_tri, d_tri_count, d_records);
  D2PC_CHECK_LAUNCH();
  return D2PC_OK;
}
