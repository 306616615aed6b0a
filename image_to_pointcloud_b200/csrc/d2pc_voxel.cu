// d2pc_voxel.cu -- ax-2, voxel-grid down-sampling of each frame's emitted rows.
// No reference code exists for this step (SURVEY.md section 8a, "parity unpinned"); the frozen
// spec is Open3D's PointCloud::VoxelDownSample: on float64 copies of the float32 points,
//   vmin = min_xyz - 0.5*vs ;  idx = floor((p - vmin) / vs) per axis ;
//   one output row per occupied voxel = arithmetic mean of member points and colours.
//
// Memory plan ("representative point" scheme).  What must be looked up at random is kept small enough to live in
// the 126 MB L2; everything large is touched in streaming order:
//   table  u32[2 N]   open addressing, one 4-byte entry per slot = 8-bit fingerprint | 24-bit row index of the
//                     voxel's REPRESENTATIVE row (the row that claimed the slot).  66 MB for a 4K frame.
//   keys   u64[N]     packed voxel index of each run leader (written in row order; read back at random only when a
//                     fingerprint matches, i.e. practically only for true members of the voxel)
//   acc    u64[5 N]   per ROW accumulators [count<<32 + sum r | sum g<<32 + sum b | sum x | sum y | sum z].  A run
//                     leader first stores its own (run-merged) sums at acc[row] in row order, fences, and only then
//                     tries to claim the slot; rows that find their voxel already claimed add their sums to the
//                     representative's accumulators with 5 RED.64.  No accumulator is ever zeroed or swept.
//   flags  u8[N]      1 = this row is a representative
//   * colours are the integral 0..255 floats emit writes: their sums are exact integers, two packed
//     64-bit adds carry count, r, g and b (N < 2^24 rows keeps every 32-bit field from overflowing);
//   * coordinates are accumulated as 64-bit fixed point of (p - bmin), bmin = the frame's min_xyz, with a
//     power-of-two scale chosen per frame from the cloud's own extent E = max over axes of (bmax - bmin), so that
//     N * E * scale < 2^62: integer adds are associative, so the means are deterministic (run-to-run identical)
//     and within 2^-38 * E of the float64 means.  The origin is NOT vmin: vmin = bmin - vs/2 would tie the
//     quantum to the voxel size, and a voxel much larger than the cloud would then lose the means.
//   * insert: one row per lane; rows that share a voxel with their left neighbour form a run that is summed in
//     registers by a segmented warp scan (raster neighbours share voxels in smooth scenes); the run's last lane
//     probes.  A read-only probe comes first, so members of an existing voxel never write their own slot.
//   * extract: streams over the rows; representatives turn their accumulators into means and are compacted
//     (CTA scan + one atomic per CTA; the order of the output rows is unspecified, as in Open3D).
// Against the first design (64-byte hash entries, 1 GB table for a 4K frame, every access a random DRAM
// read-modify-write) the random traffic drops to 4-byte entries in an L2-resident table.
#include <stdlib.h>

#include <cmath>

#include "d2pc_device.cuh"

namespace d2pc {

constexpr unsigned long long kVoxNoKey = 0xFFFFFFFFFFFFFFFFull;
constexpr uint32_t kVoxEmptySlot = 0xFFFFFFFFu;
constexpr unsigned long long kVoxMagic = 0x64327063766f7833ull;  // "d2pcvox3"
constexpr int kVoxBits = 21;
constexpr int kVoxThreads = 256;
constexpr int kVoxPerThread = 4;
constexpr int kVoxTile = kVoxThreads * kVoxPerThread;
constexpr uint32_t kVoxMaxRows = 1u << 24;  // 24-bit row index in a slot; 32-bit packed count / colour fields

struct __align__(256) VoxHeader {
  unsigned long long magic;  // kVoxMagic once d2pc_voxel_table_init has run
  uint32_t cap;              // slots allocated
  uint32_t n_out;            // output rows of the frame being processed
  uint32_t done;             // extract CTAs finished (ticket for the final count)
  uint32_t frame_cap;        // slots used for the current frame (2 * rows, >= 1024, <= cap)
  double vmin[3];            // voxel index origin: bmin - vs/2
  double origin[3];          // fixed-point origin: bmin
  double scale;              // fixed-point scale (power of two)
  int32_t bad;               // table was not initialised
};

struct VoxTable {
  VoxHeader *hdr;
  uint32_t *slots;               // [cap]
  unsigned long long *keys;      // [rows]
  unsigned long long *acc;       // [rows][5]
  uint8_t *flags;                // [rows]
  uint32_t cap, rows;
};

inline uint32_t vox_capacity(uint32_t n_rows) {
  const unsigned long long c = 2ull * n_rows;
  return (uint32_t)(c < 1024ull ? 1024ull : c);
}
inline size_t vox_bytes(uint32_t cap, uint32_t n_rows) {
  return sizeof(VoxHeader) + align_up((size_t)cap * 4, 256) + align_up((size_t)n_rows * 8, 256) +
         align_up((size_t)n_rows * 40, 256) + align_up((size_t)n_rows, 256);
}
inline VoxTable vox_table(void *base, uint32_t cap, uint32_t n_rows) {
  VoxTable t;
  char *p = (char *)base;
  t.hdr = (VoxHeader *)p;              p += sizeof(VoxHeader);
  t.slots = (uint32_t *)p;             p += align_up((size_t)cap * 4, 256);
  t.keys = (unsigned long long *)p;    p += align_up((size_t)n_rows * 8, 256);
  t.acc = (unsigned long long *)p;     p += align_up((size_t)n_rows * 40, 256);
  t.flags = (uint8_t *)p;
  t.cap = cap;
  t.rows = n_rows;
  return t;
}

__device__ __forceinline__ unsigned long long hash_u64(unsigned long long k) {
  k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
  return k;
}

__global__ void vox_init_kernel(VoxTable t) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    t.hdr->magic = kVoxMagic;
    t.hdr->cap = t.cap;
    t.hdr->n_out = 0;
    t.hdr->done = 0;
    t.hdr->bad = 0;
  }
}

// per frame: origin, fixed-point scale, slots used for this frame
__global__ void vox_begin_kernel(VoxTable t, const uint32_t *count, const float *bounds, double vs, uint32_t *ocount,
                                 int32_t *err) {
  if (threadIdx.x != 0) return;
  VoxHeader *h = t.hdr;
  *ocount = 0;
  h->n_out = 0;
  h->done = 0;
  if (h->magic != kVoxMagic || h->cap != t.cap) { h->bad = 1; h->frame_cap = 0; *err = 2; return; }
  *err = 0;
  h->bad = 0;
  const double half = vs * 0.5;
  double ext = 0.0;
  for (int c = 0; c < 3; ++c) {
    const double bmin = (double)bounds[c];
    h->vmin[c] = bmin - half;
    h->origin[c] = bmin;
    const double e = (double)bounds[3 + c] - bmin;   // float32 bounds: finite, at most 2 * FLT_MAX
    if (e > ext) ext = e;
  }
  // N * ext * scale < 2^62  with  N <= 2^24: scale = 2^(38 - ceil(log2(ext))); each term is rounded by at most
  // 0.5 / scale = 2^(ex - 39) <= 2^-38 * ext
  int ex = 0;
  if (ext > 0.0) frexp(ext, &ex);  // ext = m * 2^ex, 0.5 <= m < 1
  h->scale = ldexp(1.0, 38 - ex);
  const unsigned long long m2 = 2ull * (unsigned long long)*count;
  h->frame_cap = (uint32_t)(m2 < 1024ull ? 1024ull : (m2 > t.cap ? t.cap : m2));
}

// empty slots and clear flags for the rows of this frame (the sizes come from the header: no host sync)
__global__ void __launch_bounds__(256) vox_clear_kernel(VoxTable t, const uint32_t *count) {
  const uint32_t cap4 = (t.hdr->frame_cap + 3u) / 4u, fl16 = (*count + 15u) / 16u;
  uint4 *s4 = reinterpret_cast<uint4 *>(t.slots), *f4 = reinterpret_cast<uint4 *>(t.flags);
  const uint32_t stride = gridDim.x * blockDim.x;
  const uint64_t pol_keep = l2_policy(false, true);   // the slots should still be in L2 when the claims arrive
  const float e = __uint_as_float(kVoxEmptySlot);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < cap4; i += stride)
    stg_f4_pol(reinterpret_cast<float *>(s4 + i), make_float4(e, e, e, e), pol_keep);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < fl16; i += stride) f4[i] = make_uint4(0u, 0u, 0u, 0u);
}

// L2 residency: the 4-byte slot table (66 MB for a 4K frame) is what is probed at random and must stay in the
// 126 MB L2; the keys and accumulators (8 + 40 bytes per row) stream through and would push it out (ncu: 70% of the
// claim kernel's CAS sectors missed L2).  Slots are cleared evict-last, streamed arrays are touched evict-first.
__device__ __forceinline__ float ldg_f32_pol(const float *p, uint64_t pol) {
  float v;
  asm volatile("ld.global.nc.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(v) : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ void red_add_u64_pol(unsigned long long *p, unsigned long long v, uint64_t pol) {
  asm volatile("red.global.add.L2::cache_hint.u64 [%0], %1, %2;" :: "l"(p), "l"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ unsigned long long ld_u64_pol(const unsigned long long *p, uint64_t pol) {
  unsigned long long v;
  asm volatile("ld.global.L2::cache_hint.u64 %0, [%1], %2;" : "=l"(v) : "l"(p), "l"(pol) : "memory");
  return v;
}
__device__ __forceinline__ void st_u64_pol(unsigned long long *p, unsigned long long v, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.u64 [%0], %1, %2;" :: "l"(p), "l"(v), "l"(pol) : "memory");
}

struct VoxRun {
  unsigned long long key;
  unsigned long long cnt_r, g_b, sx, sy, sz;
};

__device__ __forceinline__ uint32_t ld_slot(const uint32_t *p) {
  uint32_t v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long ld_key(const unsigned long long *p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

__device__ __forceinline__ void vox_publish(const VoxTable &t, const VoxRun &r, uint32_t row, uint64_t pol) {
  unsigned long long *a = t.acc + 5 * (size_t)row;
  st_u64_pol(a + 0, r.cnt_r, pol); st_u64_pol(a + 1, r.g_b, pol); st_u64_pol(a + 2, r.sx, pol);
  st_u64_pol(a + 3, r.sy, pol); st_u64_pol(a + 4, r.sz, pol);
  st_u64_pol(t.keys + row, r.key, pol);
}
__device__ __forceinline__ void vox_add(const VoxTable &t, const VoxRun &r, uint32_t rep) {
  unsigned long long *a = t.acc + 5 * (size_t)rep;
  atomicAdd(a + 0, r.cnt_r);
  atomicAdd(a + 1, r.g_b);
  atomicAdd(a + 2, r.sx);
  atomicAdd(a + 3, r.sy);
  atomicAdd(a + 4, r.sz);
}

// The run leaders a lane holds (NR rows, `act` = this one leads a run; their sums and keys are already published
// and fenced): claim each voxel's slot or add the run's sums to the representative that holds it.  The NR probe
// chains are interleaved (claims together, key reads of fingerprint matches together), so a lane has NR
// independent L2 round trips in flight.
// s_sums (optional): the lane's own run sums as [NR][5][kVoxThreads] in shared memory (the fused insert kernel keeps
// them there: a member row then needs no third round trip to fetch what it is about to add).
template <int NR>
__device__ __forceinline__ void vox_claim(const VoxTable &t, uint32_t frame_cap, const unsigned long long (&key)[NR],
                                          const uint32_t (&row)[NR], const bool (&act)[NR],
                                          const unsigned long long *s_sums = nullptr) {
  uint32_t slot[NR], fp[NR], e[NR];
  bool todo[NR];
  const uint64_t pol_stream = l2_policy(true, false);
#pragma unroll
  for (int h = 0; h < NR; ++h) {
    const unsigned long long hh = hash_u64(key[h]);
    fp[h] = (uint32_t)(hh & 0xFFu) << 24;
    slot[h] = (uint32_t)(((hh >> 32) * (unsigned long long)frame_cap) >> 32);
    todo[h] = act[h];
  }
  while (true) {
    bool any = false;
#pragma unroll
    for (int h = 0; h < NR; ++h) any = any || todo[h];
    if (!any) break;
#pragma unroll
    for (int h = 0; h < NR; ++h)
      if (todo[h]) e[h] = atomicCAS(t.slots + slot[h], kVoxEmptySlot, fp[h] | row[h]);   // (atom.cas takes no cache hint)
    unsigned long long k[NR];
    bool cmp[NR];
#pragma unroll
    for (int h = 0; h < NR; ++h) {
      cmp[h] = false;
      if (!todo[h]) continue;
      if (e[h] == kVoxEmptySlot) {  // the claim succeeded: this row represents the voxel
        t.flags[row[h]] = 1;
        todo[h] = false;
      } else if ((e[h] & 0xFF000000u) == fp[h]) {
        cmp[h] = true;
        k[h] = ld_u64_pol(t.keys + (e[h] & 0x00FFFFFFu), pol_stream);
      }
    }
#pragma unroll
    for (int h = 0; h < NR; ++h) {
      if (!todo[h]) continue;
      if (cmp[h] && k[h] == key[h]) {  // a member of that row's voxel: its own published sums go to the representative
        const unsigned long long *mine = t.acc + 5 * (size_t)row[h];
        unsigned long long *a = t.acc + 5 * (size_t)(e[h] & 0x00FFFFFFu);
        unsigned long long v[5];
#pragma unroll
        for (int c = 0; c < 5; ++c)
          v[c] = s_sums ? s_sums[(h * 5 + c) * kVoxThreads + threadIdx.x] : ld_u64_pol(mine + c, pol_stream);
#pragma unroll
        for (int c = 0; c < 5; ++c) red_add_u64_pol(a + c, v[c], pol_stream);
        todo[h] = false;
      } else {
        slot[h] = slot[h] + 1u == frame_cap ? 0u : slot[h] + 1u;
      }
    }
  }
}

__device__ __forceinline__ unsigned long long shfl_up_u64(unsigned long long v, int d) {
  return __shfl_up_sync(0xffffffffu, v, d);
}

// One row per lane, kVoxPerThread consecutive 32-row groups per warp.  Rows of a group that share a
// voxel with their left neighbour form a run; a segmented warp scan sums each run into its last
// lane, which alone touches the table.  Every lane has one independent probe in flight.
template <bool SPLIT>
__global__ void __launch_bounds__(kVoxThreads, 4) vox_insert_kernel(VoxTable t, const float *xyz, const float *rgb,
                                                                    const uint32_t *count, double vs, int32_t *err) {
  const uint32_t M = *count;
  const uint32_t tile_base = blockIdx.x * (uint32_t)kVoxTile;
  if (tile_base >= M || t.hdr->bad) return;
  const double vmin0 = t.hdr->vmin[0], vmin1 = t.hdr->vmin[1], vmin2 = t.hdr->vmin[2];
  const double org0 = t.hdr->origin[0], org1 = t.hdr->origin[1], org2 = t.hdr->origin[2];
  const double scale = t.hdr->scale;
  const uint32_t frame_cap = t.hdr->frame_cap;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const double lim = (double)(1 << kVoxBits);
  const double inv_vs = 1.0 / vs;
  const uint64_t pol_stream = l2_policy(true, false);
  __shared__ unsigned long long s_sums[SPLIT ? 1 : kVoxPerThread * 5 * kVoxThreads];   // 40 KB (fused kernel only)
  unsigned long long keys[kVoxPerThread];
  uint32_t rows[kVoxPerThread];
  bool act[kVoxPerThread];
#pragma unroll
  for (int h = 0; h < kVoxPerThread; ++h) {
    const uint32_t i = tile_base + (uint32_t)((warp * kVoxPerThread + h) * 32 + lane);
    VoxRun run;
    run.key = kVoxNoKey;  // rows past the end / rejected rows: no run
    run.cnt_r = run.g_b = run.sx = run.sy = run.sz = 0ull;
    if (i < M) {
      const float *p = xyz + 3 * (size_t)i, *c = rgb + 3 * (size_t)i;
      // the rows stream through once: evict-first, like every other streamed array of the stage
      const float x0 = ldg_f32_pol(p, pol_stream), x1 = ldg_f32_pol(p + 1, pol_stream), x2 = ldg_f32_pol(p + 2, pol_stream);
      const float c0 = ldg_f32_pol(c, pol_stream), c1 = ldg_f32_pol(c + 1, pol_stream), c2 = ldg_f32_pol(c + 2, pol_stream);
      const double o0 = (double)x0 - vmin0, o1 = (double)x1 - vmin1, o2 = (double)x2 - vmin2;
      // floor((p - vmin) / vs): correctly rounded quotient from the reciprocal (d2pc_math.h).  The unguarded form is
      // enough here: offsets are >= 0; a quotient so small that the residual steps underflow floors to 0 either way,
      // and a non-finite offset gives NaN, which fails the range test below like the IEEE quotient (inf) would
      const double i0d = floor(div_by_const_fast(o0, vs, inv_vs)), i1d = floor(div_by_const_fast(o1, vs, inv_vs)),
                   i2d = floor(div_by_const_fast(o2, vs, inv_vs));
      if (i0d >= 0.0 && i0d < lim && i1d >= 0.0 && i1d < lim && i2d >= 0.0 && i2d < lim) {
        run.key = ((unsigned long long)i0d << (2 * kVoxBits)) | ((unsigned long long)i1d << kVoxBits) |
                  (unsigned long long)i2d;
        run.cnt_r = (1ull << 32) | (unsigned long long)(uint32_t)c0;
        run.g_b = ((unsigned long long)(uint32_t)c1 << 32) | (unsigned long long)(uint32_t)c2;
        run.sx = (unsigned long long)__double2ll_rn(((double)x0 - org0) * scale);
        run.sy = (unsigned long long)__double2ll_rn(((double)x1 - org1) * scale);
        run.sz = (unsigned long long)__double2ll_rn(((double)x2 - org2) * scale);
      } else {
        *err = 1;  // "voxel_size is too small." (or non-finite coordinates)
      }
    }
    // segmented inclusive scan over runs of equal keys
    const unsigned long long left = shfl_up_u64(run.key, 1);
    const bool head = (lane == 0) || (left != run.key);
    const unsigned heads = __ballot_sync(0xffffffffu, head);
    if (heads != 0xffffffffu) {  // some neighbours share a voxel (uniform branch)
      const int start = 31 - __clz(heads & (0xffffffffu >> (31 - lane)));  // first lane of my run
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const unsigned long long a0 = shfl_up_u64(run.cnt_r, d), a1 = shfl_up_u64(run.g_b, d);
        const unsigned long long a2 = shfl_up_u64(run.sx, d), a3 = shfl_up_u64(run.sy, d), a4 = shfl_up_u64(run.sz, d);
        if (lane - d >= start) { run.cnt_r += a0; run.g_b += a1; run.sx += a2; run.sy += a3; run.sz += a4; }
      }
    }
    const bool tail = (lane == 31) || ((heads >> (lane + 1)) & 1u);
    keys[h] = run.key;
    rows[h] = i;
    act[h] = tail && run.key != kVoxNoKey;
    if (act[h]) {
      vox_publish(t, run, i, pol_stream);   // in row order: a streaming write
      if (!SPLIT) {
        unsigned long long *m = s_sums + (size_t)(h * 5) * kVoxThreads + threadIdx.x;
        m[0] = run.cnt_r; m[kVoxThreads] = run.g_b; m[2 * kVoxThreads] = run.sx; m[3 * kVoxThreads] = run.sy;
        m[4 * kVoxThreads] = run.sz;
      }
    }
    else if (SPLIT && i < M) st_u64_pol(t.keys + i, kVoxNoKey, pol_stream);   // the claim kernel reads every row's key
  }
  if (SPLIT) return;   // the table is touched by vox_claim_kernel (the kernel boundary orders the published sums)
  __threadfence();   // one fence for the lane's rows: sums and keys are in place before any row can be found
  vox_claim<kVoxPerThread>(t, frame_cap, keys, rows, act, s_sums);
}

// The table half of the insert as its own launch: the run leaders' keys come back from the keys array (a coalesced
// read) and nothing of the row's arithmetic is alive, so the kernel needs few registers and twice as many probe
// chains are in flight per SM -- the stage is a chain of L2 round trips (CAS -> key compare -> sums -> 5 RED per
// member row), not a stream.
__global__ void __launch_bounds__(kVoxThreads, 6) vox_claim_kernel(VoxTable t, const uint32_t *count) {
  const uint32_t M = *count;
  const uint32_t tile_base = blockIdx.x * (uint32_t)kVoxTile;
  if (tile_base >= M || t.hdr->bad) return;
  const uint32_t frame_cap = t.hdr->frame_cap;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned long long keys[kVoxPerThread];
  uint32_t rows[kVoxPerThread];
  bool act[kVoxPerThread];
#pragma unroll
  for (int h = 0; h < kVoxPerThread; ++h) {
    const uint32_t i = tile_base + (uint32_t)((warp * kVoxPerThread + h) * 32 + lane);
    rows[h] = i;
    keys[h] = i < M ? __ldcs(t.keys + i) : kVoxNoKey;
  }
#pragma unroll
  for (int h = 0; h < kVoxPerThread; ++h) act[h] = keys[h] != kVoxNoKey;
  vox_claim<kVoxPerThread>(t, frame_cap, keys, rows, act);
}

// streams over the rows: representatives -> means -> compacted output rows
__global__ void __launch_bounds__(kVoxThreads, 3) vox_extract_kernel(VoxTable t, const uint32_t *count, float *oxyz,
                                                                     float *orgb, int32_t *oidx, uint32_t *ocount,
                                                                     const int32_t *err) {
  __shared__ uint32_t s_warp[kVoxThreads / 32];
  __shared__ uint32_t s_base;
  const uint32_t M = *count;
  const uint32_t tile_base = blockIdx.x * (uint32_t)kVoxTile;
  if (tile_base >= M || t.hdr->bad) return;  // uniform
  const bool failed = *err != 0;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t i0 = tile_base + 4u * (uint32_t)tid;   // 4 consecutive rows per thread
  uint32_t f = 0;
  if (i0 < M) f = *reinterpret_cast<const uint32_t *>(t.flags + i0);  // rows >= M were cleared (padding to 16)
  const uint32_t mine = __popc(f & 0x01010101u);
  uint32_t incl = mine;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t y = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += y;
  }
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();
  uint32_t woff = 0, total = 0;
#pragma unroll
  for (int w = 0; w < kVoxThreads / 32; ++w) {
    const uint32_t x = s_warp[w];
    if (w < warp) woff += x;
    total += x;
  }
  if (tid == 0) s_base = (total && !failed) ? atomicAdd(&t.hdr->n_out, total) : 0u;
  __syncthreads();
  if (!failed && mine) {
    uint32_t j = s_base + woff + incl - mine;
    const double inv_scale = 1.0 / t.hdr->scale;  // power of two: exact
    const double org0 = t.hdr->origin[0], org1 = t.hdr->origin[1], org2 = t.hdr->origin[2];
    unsigned long long w[4][6];
#pragma unroll
    for (int k = 0; k < 4; ++k) {  // all loads of the thread's representatives in flight together
      if (!((f >> (8 * k)) & 1u)) continue;
      const uint32_t row = i0 + (uint32_t)k;
      const unsigned long long *a = t.acc + 5 * (size_t)row;
#pragma unroll
      for (int c = 0; c < 5; ++c) w[k][c] = __ldcg(a + c);
      w[k][5] = __ldcg(t.keys + row);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (!((f >> (8 * k)) & 1u)) continue;
      const unsigned long long cnt_r = w[k][0], g_b = w[k][1], sx = w[k][2], sy = w[k][3], sz = w[k][4], key = w[k][5];
      const double n = (double)(uint32_t)(cnt_r >> 32);   // >= 1
      // six means per row: one division (the reciprocal) and the correctly rounded quotients from it
      // (div_by_const_fast: numerators are >= 0 and finite, n is a small integer -- same bits as a / n)
      const double rn = 1.0 / n;
      float *ox = oxyz + 3 * (size_t)j, *oc = orgb + 3 * (size_t)j;
      stg_stream_f1(ox + 0, (float)(org0 + div_by_const_fast((double)(long long)sx * inv_scale, n, rn)));
      stg_stream_f1(ox + 1, (float)(org1 + div_by_const_fast((double)(long long)sy * inv_scale, n, rn)));
      stg_stream_f1(ox + 2, (float)(org2 + div_by_const_fast((double)(long long)sz * inv_scale, n, rn)));
      stg_stream_f1(oc + 0, (float)div_by_const_fast((double)(uint32_t)cnt_r, n, rn));
      stg_stream_f1(oc + 1, (float)div_by_const_fast((double)(uint32_t)(g_b >> 32), n, rn));
      stg_stream_f1(oc + 2, (float)div_by_const_fast((double)(uint32_t)g_b, n, rn));
      if (oidx) {
        oidx[3 * (size_t)j + 0] = (int32_t)(key >> (2 * kVoxBits));
        oidx[3 * (size_t)j + 1] = (int32_t)((key >> kVoxBits) & ((1u << kVoxBits) - 1u));
        oidx[3 * (size_t)j + 2] = (int32_t)(key & ((1u << kVoxBits) - 1u));
      }
      ++j;
    }
  }
  // the last CTA with work publishes the count
  __syncthreads();
  if (tid == 0) {
    __threadfence();
    const uint32_t ticket = atomicAdd(&t.hdr->done, 1u);
    if (ticket == (M + kVoxTile - 1) / kVoxTile - 1) {
      *ocount = failed ? 0u : *reinterpret_cast<volatile uint32_t *>(&t.hdr->n_out);
    }
  }
}

}  // namespace d2pc

using namespace d2pc;

extern "C" int d2pc_voxel_table_bytes(const D2pcConfig *cfg, size_t *bytes) {
  int rc = validate_config(cfg);
  if (rc) return rc;
  if (!bytes) return D2PC_ERR_INVALID_ARGUMENT;
  const Geom g = make_geom(*cfg);
  if (g.N >= kVoxMaxRows) return D2PC_ERR_UNSUPPORTED;
  *bytes = vox_bytes(vox_capacity(g.N), g.N);
  return D2PC_OK;
}

extern "C" int d2pc_voxel_table_init(const D2pcConfig *cfg, void *d_table, size_t table_bytes, void *stream) {
  int rc = validate_config(cfg);
  if (rc) return rc;
  if (!d_table || ((uintptr_t)d_table & 255u) != 0) return D2PC_ERR_INVALID_ARGUMENT;
  const Geom g = make_geom(*cfg);
  if (g.N >= kVoxMaxRows) return D2PC_ERR_UNSUPPORTED;
  const uint32_t cap = vox_capacity(g.N);
  if (table_bytes < vox_bytes(cap, g.N)) return D2PC_ERR_WORKSPACE_TOO_SMALL;
  vox_init_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(vox_table(d_table, cap, g.N));
  D2PC_CHECK_LAUNCH();
  return D2PC_OK;
}

extern "C" int d2pc_voxel_enqueue(const D2pcConfig *cfg, double voxel_size, const float *d_xyz,
                                  const float *d_rgb, const uint32_t *d_count, const float *d_bounds,
                                  void *d_table, size_t table_bytes, float *d_vox_xyz, float *d_vox_rgb,
                                  int32_t *d_vox_idx, uint32_t *d_vox_count, int32_t *d_vox_error,
                                  void *stream) {
  int rc = validate_config(cfg);
  if (rc) return rc;
  if (!(std::isfinite(voxel_size) && voxel_size > 0.0)) return D2PC_ERR_INVALID_ARGUMENT;
  if (!d_xyz || !d_rgb || !d_count || !d_bounds || !d_table || !d_vox_xyz || !d_vox_rgb || !d_vox_count ||
      !d_vox_error)
    return D2PC_ERR_INVALID_ARGUMENT;
  if (((uintptr_t)d_table & 255u) != 0) return D2PC_ERR_INVALID_ARGUMENT;
  const Geom g = make_geom(*cfg);
  if (g.N >= kVoxMaxRows) return D2PC_ERR_UNSUPPORTED;
  const uint32_t cap = vox_capacity(g.N);
  if (table_bytes < vox_bytes(cap, g.N)) return D2PC_ERR_WORKSPACE_TOO_SMALL;
  cudaStream_t st = (cudaStream_t)stream;
  VoxTable t = vox_table(d_table, cap, g.N);
  const uint32_t tiles = (g.N + kVoxTile - 1) / kVoxTile;
  for (int b = 0; b < cfg->batch; ++b) {
    const size_t ro = (size_t)b * g.N * 3;
    vox_begin_kernel<<<1, 32, 0, st>>>(t, d_count + b, d_bounds + 6 * b, voxel_size, d_vox_count + b,
                                       d_vox_error + b);
    D2PC_CHECK_LAUNCH();
    vox_clear_kernel<<<148 * 4, 256, 0, st>>>(t, d_count + b);
    D2PC_CHECK_LAUNCH();
    // One fused insert kernel by default.  Publishing and claiming as two launches (the claim kernel then runs at
    // 6 CTAs per SM instead of 4) was measured: 363 / 307 / 312 us against 338 / 294 / 266 us fused (4K frame, smooth
    // scene 5 mm / uniform depth 5 mm / scene 5 cm) once the streamed arrays carry evict-first hints.
    const char *se = getenv("D2PC_VOX_SPLIT");  // measurement aid: "1" = publish + claim as two launches
    if (!(se && atoi(se) != 0)) {
      vox_insert_kernel<false><<<tiles, kVoxThreads, 0, st>>>(t, d_xyz + ro, d_rgb + ro, d_count + b, voxel_size,
                                                              d_vox_error + b);
    } else {
      vox_insert_kernel<true><<<tiles, kVoxThreads, 0, st>>>(t, d_xyz + ro, d_rgb + ro, d_count + b, voxel_size,
                                                             d_vox_error + b);
      D2PC_CHECK_LAUNCH();
      vox_claim_kernel<<<tiles, kVoxThreads, 0, st>>>(t, d_count + b);
    }
    D2PC_CHECK_LAUNCH();
    vox_extract_kernel<<<tiles, kVoxThreads, 0, st>>>(t, d_count + b, d_vox_xyz + ro, d_vox_rgb + ro,
                                                        d_vox_idx ? d_vox_idx + ro : nullptr, d_vox_count + b,
                                                        d_vox_error + b);
    D2PC_CHECK_LAUNCH();
  }
  return D2PC_OK;
}
