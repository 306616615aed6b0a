/*
 * d2pc.h -- C ABI of libd2pc.so: the B200 (sm_100a) depth-map -> coloured point-cloud stage.
 *
 * What this replaces.  The reference has no FFI or plugin boundary for this path: the stage is
 * one Python function, depth_to_point_cloud(image, depth, density, invert, depth_scale, smooth,
 * smooth_ksize, fov) -> (points f32[N,3], colors f32[N,3])   (reference backend/app.py:174-250),
 * called once per request at backend/app.py:468-476.  The drop-in is therefore a Python function
 * of the same name and signature (image_to_pointcloud_b200.depth_to_point_cloud) that rebinds
 * that name; the entry points below are what that function binds with ctypes, and what any
 * other host (C, C++, cgo, JNI, N-API) would bind.  INTEGRATION.md shows the stub.
 *
 * Conventions
 *  - plain C types only; every pointer named d_* is a DEVICE pointer owned by the caller
 *    (torch tensors in the Python host), including the workspace.  The library allocates
 *    nothing, keeps no global state and never synchronises the host: every call only enqueues
 *    kernels on `stream` (a cudaStream_t passed as void*).  Re-entrant per (device, stream).
 *  - return value: 0 = D2PC_OK, otherwise a D2PC_ERR_* code; nothing is thrown across the ABI.
 *    d2pc_error_string() gives the text.  The Python host raises on non-zero, so the reference's
 *    error convention (raise -> pipeline marks the job "error", app.py:248-250,561-565) holds.
 *  - a "frame" is one (image, depth) pair.  A call processes `batch` frames that share geometry
 *    and knobs; frames are independent (own percentiles, own output slot, no cross-frame state:
 *    the reference function is pure), which is also the multi-GPU sharding unit.
 *
 * Reference step -> entry point
 *   a1 resize (app.py:186-188), a2 non-finite repair (:191-196), a3 percentiles (:197-199),
 *   a4 clip+normalise (:200-204), a5 invert (:205-206)       -> d2pc_stats_enqueue
 *                                                               (+ d2pc_stats_fallback_enqueue)
 *   a7 intrinsics (:216-223), a8 stride (:225-226)            -> D2pcConfig fields (host computes
 *                                                               cx, cy, f exactly as the reference)
 *   a9 back-projection (:228-237), a10 colour gather (:239-244),
 *   a11 emission (:246), ax-1 depth-range mask + compaction   -> d2pc_emit_enqueue
 *   ax-2 voxel-grid down-sampling (north-star extension)      -> d2pc_voxel_enqueue
 *   f1 refine_point_cloud (:252-269, Open3D SOR)               -> d2pc_sor_enqueue
 *   f5 density clustering (Open3D cluster_dbscan,
 *      remove_radius_outlier)                                  -> d2pc_dbscan_enqueue, d2pc_radius_outlier_enqueue
 *   f3 preview stride (:495-506), save_xyz/las/ply (:329-389) -> d2pc_preview_rows_enqueue,
 *                                                               d2pc_xyz_text_*, d2pc_las_records_enqueue,
 *                                                               d2pc_ply_records_enqueue
 *   n1 point normals (the mesh builder's first step, :271-308) -> d2pc_normals_enqueue
 *   m1 lattice mesh (our own spec; the reference meshes with
 *      Poisson / BPA, :271-308)                                -> d2pc_grid_mesh_enqueue,
 *                                                               d2pc_ply_face_records_enqueue
 *   m2 mesh simplification by vertex clustering (the reference
 *      decimates its mesh for the preview, :271-308, 508-535)  -> d2pc_mesh_simplify_enqueue
 */
#ifndef D2PC_H_
#define D2PC_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define D2PC_ABI_VERSION 1

enum {
  D2PC_OK = 0,
  D2PC_ERR_INVALID_ARGUMENT = 1, /* bad geometry / null pointer / unsupported knob          */
  D2PC_ERR_WORKSPACE_TOO_SMALL = 2,
  D2PC_ERR_CUDA = 3,             /* a CUDA runtime call or launch failed (see error_string)  */
  D2PC_ERR_UNSUPPORTED = 4       /* valid reference input this build does not implement yet  */
};

/* per-frame status word written by the stats kernels (workspace, see d2pc_frame_status) */
enum {
  D2PC_FRAME_PENDING = 0,
  D2PC_FRAME_READY = 1,          /* normalisation parameters are final; emit may run         */
  D2PC_FRAME_NEEDS_FALLBACK = 2  /* fast selection declined (non-finite values, bracket miss,
                                    candidate overflow): run d2pc_stats_fallback_enqueue     */
};

/* normalisation branch taken for a frame (reference app.py:197-204) */
enum {
  D2PC_BRANCH_PCT = 0,    /* p98 > p2: float64 clip/normalise chain                          */
  D2PC_BRANCH_MINMAX = 1, /* percentiles degenerate, min < max: float32 chain                */
  D2PC_BRANCH_ZEROS = 2   /* constant (or NaN-poisoned) map: d = 0                           */
};

/* Geometry and knobs shared by all frames of a call.  Plain old data, passed by pointer. */
typedef struct D2pcConfig {
  int32_t batch;        /* frames in this call (>= 1)                                        */
  int32_t img_h, img_w; /* H, W of the image = size of the output grid                      */
  int32_t img_c;        /* image channels: 3 or 4 (BGR / BGRA, app.py:240-242); 1 = grey ->
                           colour [128,128,128] (app.py:243-244)                            */
  int32_t dep_h, dep_w; /* h, w of the depth map; != (H, W) -> bilinear resize (app.py:187) */
  int32_t step;         /* sampling stride: 4 / 2 / 1 for low / medium / high (app.py:226)  */
  int32_t invert;       /* app.py:205                                                       */
  double depth_scale;   /* app.py:233                                                       */
  double cx, cy, f;     /* intrinsics, computed by the host as app.py:219-223               */
  /* ax-1 depth-range mask (extension; off = keep every point like the reference) */
  int32_t use_z_range;  /* 0 / 1                                                            */
  float z_min, z_max;   /* keep iff z_min <= z32 <= z_max on the emitted float32 z          */
  int32_t drop_nonfinite; /* 1: also drop points whose (resized) depth was NaN/inf          */
  int32_t want_bounds;  /* 1: emit also reduces per-frame min/max of kept xyz (for voxels,
                           LAS offsets app.py:352 and GIS bounds app.py:394-399)            */
  int32_t force_fallback; /* test hook: 1 = stats marks every frame NEEDS_FALLBACK          */
} D2pcConfig;

/* Normalisation parameters of one frame as the device computed them (debug / tests). */
typedef struct D2pcFrameParams {
  double p2, p98;       /* the two scalars of app.py:197-199 (after the min/max fallback)    */
  double den;           /* (p98 - p2) + 1e-6                                                 */
  double inv_den;       /* correctly rounded 1/den                                           */
  float lo32, hi32, den32; /* float32 operands of the MINMAX branch                         */
  float median;         /* np.nanmedian replacement value (valid if n_nonfinite > 0)        */
  int32_t branch;       /* D2PC_BRANCH_*                                                    */
  int32_t status;       /* D2PC_FRAME_*                                                     */
  uint32_t n_nonfinite; /* NaN or +-inf in the (resized) map                                */
  uint32_t n_nan;
  uint32_t n_cand[2];   /* candidates collected for the 2% / 98% brackets (fast path)       */
  uint32_t reserved[2];
} D2pcFrameParams;

int d2pc_abi_version(void);
const char *d2pc_error_string(int code);
/* text of the last CUDA error seen by this thread inside the library ("" if none) */
const char *d2pc_last_cuda_error(void);

/* Bytes of workspace needed for cfg (depends on batch and geometry only). */
int d2pc_workspace_bytes(const D2pcConfig *cfg, size_t *bytes);

/* a1..a5: exact 2nd/98th percentile statistics of every frame's (virtually resized) depth map
 * and the frame's normalisation parameters, entirely on the device.
 *   d_depth  float32 [batch, dep_h, dep_w]
 * Fast path: sample -> brackets -> one streaming pass (counts + candidates) -> exact select.
 * Frames it cannot finish exactly are marked D2PC_FRAME_NEEDS_FALLBACK. */
int d2pc_stats_enqueue(const D2pcConfig *cfg, const float *d_depth, void *d_workspace,
                       size_t workspace_bytes, void *stream);

/* Exact, input-agnostic selection (multi-pass radix select, nanmedian repair) for every frame
 * whose status is NEEDS_FALLBACK; no-op kernels for the others. */
int d2pc_stats_fallback_enqueue(const D2pcConfig *cfg, const float *d_depth, void *d_workspace,
                                size_t workspace_bytes, void *stream);

/* Copies the per-frame status words (int32 [batch]) to a device buffer the host can read back
 * with one small memcpy; d_any_fallback (int32 [1]) is set to 1 if any frame needs it. */
int d2pc_frame_status(const D2pcConfig *cfg, const void *d_workspace, int32_t *d_status,
                      int32_t *d_any_fallback, void *stream);

/* Copies the per-frame parameter blocks to d_params (D2pcFrameParams [batch]). */
int d2pc_frame_params(const D2pcConfig *cfg, const void *d_workspace, D2pcFrameParams *d_params,
                      void *stream);

/* a4..a11 (+ ax-1): fused resize / repair / normalise / invert / back-project / colour gather /
 * mask / ordered compaction / packing.
 *   d_bgr    uint8  [batch, H, W, img_c]           (may be NULL when img_c == 1)
 *   d_xyz    float32 [batch, N, 3], d_rgb likewise, N = ceil(H/step) * ceil(W/step)
 *   d_count  uint32 [batch]   rows emitted per frame (== N unless a mask is active)
 *   d_bounds float32 [batch, 6] (min x,y,z, max x,y,z) if cfg->want_bounds, else may be NULL */
int d2pc_emit_enqueue(const D2pcConfig *cfg, const float *d_depth, const uint8_t *d_bgr,
                      void *d_workspace, size_t workspace_bytes, float *d_xyz, float *d_rgb,
                      uint32_t *d_count, float *d_bounds, void *stream);

/* The whole path (d2pc_stats_enqueue + d2pc_frame_status + d2pc_emit_enqueue) of a batch as ONE software
 * pipeline over sub-batches of `sub_batch` frames (csrc/d2pc_path.cu): the statistics of sub-batch k+1 run on
 * an auxiliary high-priority stream while the emit of sub-batch k streams its rows out, with L2 eviction hints
 * such that every depth map (or materialised resized map) is read from HBM once.  Results are identical to
 * the two-phase calls.  Frames the fast statistics cannot finish exactly are left out and flagged in d_status /
 * *d_any_fallback (either may be NULL) exactly like d2pc_frame_status; the host then runs the two-phase calls
 * with d2pc_stats_fallback_enqueue in between (python: FrameEngine.process).
 *   D2pcPath     opaque handle: the auxiliary stream, the events of the fork / join and a cached CUDA graph.
 *                The one exception to "the library allocates nothing": created and destroyed by the caller,
 *                bound to the device that was current at creation, used by one host thread at a time.
 *   sub_batch    frames per pipeline stage (<= 0 or >= batch: one stage, no overlap)
 *   lookahead    sub-batches the statistics may run ahead of the emit (>= 1)
 *   flags        D2PC_PATH_GRAPH: capture the step into a CUDA graph once and replay it while all arguments
 *                repeat (steady-state batches); D2PC_PATH_NO_OVERLAP / D2PC_PATH_NO_L2_HINTS: measurement aids */
typedef struct D2pcPath D2pcPath;
#define D2PC_PATH_GRAPH 1
#define D2PC_PATH_NO_OVERLAP 2
#define D2PC_PATH_NO_L2_HINTS 4
#define D2PC_PATH_ORDERED 8
int d2pc_path_create(D2pcPath **path);
void d2pc_path_destroy(D2pcPath *path);
int d2pc_path_enqueue(D2pcPath *path, const D2pcConfig *cfg, const float *d_depth, const uint8_t *d_bgr,
                      void *d_workspace, size_t workspace_bytes, float *d_xyz, float *d_rgb, uint32_t *d_count,
                      float *d_bounds, int32_t *d_status, int32_t *d_any_fallback, int32_t sub_batch,
                      int32_t lookahead, int32_t flags, void *stream);

/* measurement aid: byte offset in the workspace of the persistent kernel's per-frame trace (8 x uint64 ns per frame:
 * first scan tile, last scan tile, selection start / end of bracket 0 and 1, first emit tile, last emit tile) */
int d2pc_path_trace_offset(const D2pcConfig *cfg, size_t *offset);

/* a6 + a9..a11: the same emission with the optional smoothing of app.py:208-214 switched on:
 * cv2.GaussianBlur(d, (k, k), 0) on the normalised (and inverted) map before the back-projection.
 *   ksize      k = max(3, smooth_ksize // 2 * 2 + 1), odd, <= D2PC_MAX_SMOOTH_KSIZE
 *   h_kernel   HOST pointer to k float64 coefficients = cv2.getGaussianKernel(k, 0, CV_64F)
 *   d_scratch  device scratch of d2pc_smooth_scratch_bytes() bytes (two float64 maps per frame)
 * Arithmetic follows OpenCV 4.13's float64 separable filter (rows with FMA in the vector body and
 * plain multiply-add in the last W%4 columns, then symmetric column sums; BORDER_REFLECT_101), so
 * percentile-branch frames are bit-exact for k <= 9; the float32 (min/max) branch is within 1e-6. */
#define D2PC_MAX_SMOOTH_KSIZE 255
int d2pc_smooth_scratch_bytes(const D2pcConfig *cfg, size_t *bytes);
int d2pc_emit_smooth_enqueue(const D2pcConfig *cfg, const float *d_depth, const uint8_t *d_bgr,
                             void *d_workspace, size_t workspace_bytes, int32_t ksize,
                             const double *h_kernel, void *d_scratch, size_t scratch_bytes,
                             float *d_xyz, float *d_rgb, uint32_t *d_count, float *d_bounds,
                             void *stream);

/* f2 depth preview (reference create_depth_preview, app.py:124-153): the same robust normalisation
 * on the UN-resized depth map (call d2pc_stats_enqueue first with img_h/img_w == dep_h/dep_w), then
 * (d * 255).astype(uint8) and the colour-map lookup.
 *   d_lut_bgr  uint8 [256, 3] colour map (COLORMAP_PLASMA, BGR)
 *   d_out_bgr  uint8 [batch, h, w, 3]
 * PNG encoding and the optional INTER_AREA down-scale stay on the host. */
int d2pc_preview_enqueue(const D2pcConfig *cfg, const float *d_depth, void *d_workspace,
                         size_t workspace_bytes, const uint8_t *d_lut_bgr, uint8_t *d_out_bgr,
                         void *stream);

/* ax-2 voxel-grid down-sampling of each frame's emitted rows (Open3D VoxelDownSample semantics:
 * vmin = min_xyz - vs/2, idx = floor((p - vmin)/vs) on float64 copies, mean of members).
 *   voxel_size    finite and > 0 (else D2PC_ERR_INVALID_ARGUMENT before any launch)
 *   d_xyz/d_rgb/d_count/d_bounds  outputs of d2pc_emit_enqueue (want_bounds = 1), row stride N;
 *                 colours must be the integral 0..255 values emit writes (their sums are kept exact)
 *   d_table       scratch of d2pc_voxel_table_bytes() bytes, 256-byte aligned, on which
 *                 d2pc_voxel_table_init() has run with a config of the same rows per frame N: a table of
 *                 4-byte slots (8-bit fingerprint | 24-bit row of the voxel's representative row, small enough
 *                 to stay in L2), and per-row keys, accumulators and flags that are only touched in row order
 *                 (csrc/d2pc_voxel.cu).  The layout depends on N, so initialise again whenever the config's N
 *                 changes (another density); otherwise the frames fail with error 2.  Cleared per frame by the
 *                 call itself.
 *   d_vox_xyz/rgb float32 [batch, N, 3]; d_vox_idx int32 [batch, N, 3] or NULL;
 *   d_vox_count   uint32 [batch]; d_vox_error int32 [batch] (1 = index overflow, >= 2^21;
 *                 2 = table not initialised)
 * Coordinates are summed as 64-bit fixed point of (p - min_xyz), scaled to the cloud's extent
 * E = max over axes of (max_xyz - min_xyz): the means are deterministic and within 2^-38 * E (plus the
 * float32 rounding of the result) of the float64 means, whatever the voxel size.  Colour means are exact
 * (correctly rounded quotients of exact integer sums).  Frames of 2^24 rows or more return
 * D2PC_ERR_UNSUPPORTED. */
int d2pc_voxel_table_bytes(const D2pcConfig *cfg, size_t *bytes);
int d2pc_voxel_table_init(const D2pcConfig *cfg, void *d_table, size_t table_bytes, void *stream);
int d2pc_voxel_enqueue(const D2pcConfig *cfg, double voxel_size, const float *d_xyz,
                       const float *d_rgb, const uint32_t *d_count, const float *d_bounds,
                       void *d_table, size_t table_bytes, float *d_vox_xyz, float *d_vox_rgb,
                       int32_t *d_vox_idx, uint32_t *d_vox_count, int32_t *d_vox_error,
                       void *stream);

/* f3 -- byte layouts of the reference's writers and preview (backend/app.py:310-389, 495-506), produced on
 * the device from ONE frame's emitted rows (d_xyz / d_rgb point at that frame's slot, d_count at its row
 * count; capacity_rows = N bounds the launch).  Headers and file I/O stay on the host.
 *
 * preview rows (app.py:495-500): points[::stride], stride = max(1, n // max_preview) when n > max_preview.
 *   d_out_xyz/rgb float32 [out_capacity_rows, 3] (2 * max_preview rows always suffice); d_out_count uint32 [1] */
int d2pc_preview_rows_enqueue(const float *d_xyz, const float *d_rgb, const uint32_t *d_count,
                              uint32_t max_preview, float *d_out_xyz, float *d_out_rgb,
                              uint32_t out_capacity_rows, uint32_t *d_out_count, void *stream);

/* XYZ ASCII (save_xyz, app.py:379-389): one line f"{x:.6f} {y:.6f} {z:.6f} {int(r)} {int(g)} {int(b)}\n" per
 * row, byte-identical to Python's formatting of numpy.float32 values.  Two steps because the size is data
 * dependent: measure (per-tile byte counts + scan -> *d_text_bytes, *d_error = 1 if a value cannot be
 * formatted: |coordinate| >= 2^44, non-finite colour), then write into a buffer of at least that size. */
int d2pc_xyz_text_scratch_bytes(uint32_t capacity_rows, size_t *bytes);
int d2pc_xyz_text_measure_enqueue(const float *d_xyz, const float *d_rgb, const uint32_t *d_count,
                                  uint32_t capacity_rows, void *d_scratch, size_t scratch_bytes,
                                  unsigned long long *d_text_bytes, int32_t *d_error, void *stream);
int d2pc_xyz_text_write_enqueue(const float *d_xyz, const float *d_rgb, const uint32_t *d_count,
                                uint32_t capacity_rows, const void *d_scratch, size_t scratch_bytes,
                                const unsigned long long *d_text_bytes, const int32_t *d_error, char *d_text,
                                size_t text_capacity, void *stream);

/* min / max x, y, z of the rows (float(points[:, k].min()) ..., app.py:352, 394-399) for callers that did not
 * ask emit for its fused bounds: d_scratch6 uint32 [6], d_bounds6 float32 [6] = min x,y,z, max x,y,z
 * (the d_bounds layout of emit; NaN for an empty cloud). */
int d2pc_rows_bounds_enqueue(const float *d_xyz, const uint32_t *d_count, uint32_t capacity_rows,
                             uint32_t *d_scratch6, float *d_bounds6, void *stream);

/* LAS 1.2 point format 2 records (save_las, app.py:343-377), 26 bytes each: X/Y/Z = int32(np.round((x -
 * offset) / scale)) with offset = the frame's min x/y/z (d_bounds of emit, want_bounds = 1), colours
 * uint16(clip(c, 0, 255)) * 256, all other fields 0.  d_int_minmax int32 [6] = min X,Y,Z, max X,Y,Z (for the
 * header); *d_error = 1 if a scaled coordinate leaves int32.  d_records must be 16-byte aligned. */
int d2pc_las_records_enqueue(const float *d_xyz, const float *d_rgb, const uint32_t *d_count,
                             uint32_t capacity_rows, const float *d_bounds, double scale, uint8_t *d_records,
                             int32_t *d_int_minmax, int32_t *d_error, void *stream);

/* Binary little-endian PLY vertices as Open3D writes them (save_ply, app.py:329-341), 27 bytes each:
 * float64 x, y, z; uchar red, green, blue = round(clamp(float32(c / 255), 0, 1) * 255). */
int d2pc_ply_records_enqueue(const float *d_xyz, const float *d_rgb, const uint32_t *d_count,
                             uint32_t capacity_rows, uint8_t *d_records, void *stream);

/* The same vertices for a cloud with normals, 51 bytes each in Open3D's property order: float64 x, y, z, nx, ny, nz;
 * uchar red, green, blue.  d_normals float64 [capacity_rows, 3] (d2pc_normals_enqueue); d_records 16-byte aligned. */
int d2pc_ply_normal_records_enqueue(const float *d_xyz, const double *d_normals, const float *d_rgb,
                                    const uint32_t *d_count, uint32_t capacity_rows, uint8_t *d_records,
                                    void *stream);

/* f1 -- statistical outlier removal (refine_point_cloud, app.py:252-269: Open3D remove_statistical_outlier(
 * nb_neighbors=20, std_ratio=2.0)) on ONE frame's rows: exact k-nearest neighbours (the point itself
 * included, float64 distances) through a uniform grid, avg[i] = mean of the k distances, keep
 * 0 < avg[i] < mean(avg) + std_ratio * std(avg) (Bessel-corrected, Open3D's definitions), kept rows in order.
 *   d_bounds     float32 [6] min/max of the rows (emit want_bounds = 1, or d2pc_rows_bounds_enqueue)
 *   d_scratch    d2pc_sor_scratch_bytes(capacity_rows) bytes, 256-byte aligned
 *   d_out_xyz/rgb float32 [capacity_rows, 3] (d_rgb / d_out_rgb may both be NULL); d_out_index uint32
 *                [capacity_rows] source row of every kept row, or NULL; d_out_count uint32 [1]
 *   d_stats      float64 [4] = cloud mean, standard deviation, threshold, N; or NULL
 *   nb_neighbors 1..64 */
int d2pc_sor_scratch_bytes(uint32_t capacity_rows, size_t *bytes);
int d2pc_sor_enqueue(const float *d_xyz, const float *d_rgb, const uint32_t *d_count, uint32_t capacity_rows,
                     const float *d_bounds, int32_t nb_neighbors, double std_ratio, void *d_scratch,
                     size_t scratch_bytes, float *d_out_xyz, float *d_out_rgb, uint32_t *d_out_index,
                     uint32_t *d_out_count, double *d_stats, void *stream);

/* f5 -- density clustering of ONE cloud (Open3D ClusterDBSCAN and RemoveRadiusOutliers; spec in
 * oracle/d2pc_cluster_oracle.py).  Point j is a neighbour of point i when d2(i, j) < eps * eps (strict), d2 summed
 * axis by axis in float64 from the float32 rows; the point itself is a neighbour.  A uniform grid of cell side
 * eps / 2 * (1 + 2^-20) holds the rows, so every neighbour lies in the 5 x 5 x 5 cells around a row's own cell.
 *   d_bounds       float32 [6] min/max of the rows (d2pc_rows_bounds_enqueue)
 *   d_scratch      d2pc_cluster_scratch_bytes(capacity_rows) bytes, 256-byte aligned
 *   d_out_xyz/rgb  float32 [capacity_rows, 3] kept rows in input order (d_rgb / d_out_rgb may both be NULL);
 *                  d_out_index uint32 [capacity_rows] their source rows, or NULL
 *   d_out_counts   uint32 [4] = kept rows, error bits (D2PC_CLUSTER_ERR_*), clusters (DBSCAN only), 0
 * The error bits are set on the device: a row with a non-finite coordinate; an eps so small that an axis of the
 * bounding box needs 1048574 cells or more (the grid cannot hold the cloud: the call refuses it rather than return
 * a wrong result); an exhausted loop bound (an internal failure, never expected).  Any error leaves the other
 * outputs undefined.  No floating-point atomics: the result repeats bit for bit.  Argument errors are returned
 * before any launch; the call does not synchronise. */
enum { D2PC_CLUSTER_ERR_NONFINITE = 1, D2PC_CLUSTER_ERR_GRID = 2, D2PC_CLUSTER_ERR_BOUND = 4 };
int d2pc_cluster_scratch_bytes(uint32_t capacity_rows, size_t *bytes);
/* Row i is kept iff it has more than nb_points neighbours within radius (itself counted).  nb_points >= 1, radius
 * finite and > 0 with radius * radius > 0. */
int d2pc_radius_outlier_enqueue(const float *d_xyz, const float *d_rgb, const uint32_t *d_count,
                                uint32_t capacity_rows, const float *d_bounds, int32_t nb_points, double radius,
                                void *d_scratch, size_t scratch_bytes, float *d_out_xyz, float *d_out_rgb,
                                uint32_t *d_out_index, uint32_t *d_out_counts, void *stream);
/* DBSCAN: a row is core when it has at least min_points neighbours; clusters are the connected components of the
 * cores under the neighbour relation, numbered 0, 1, ... by their lowest core row; a non-core row takes the lowest
 * cluster among its core neighbours, else -1.
 *   d_out_labels   int32 [capacity_rows]; d_out_sizes uint32 [capacity_rows], the rows of every cluster
 *   min_size       with d_out_xyz set, the rows of clusters of at least min_size rows are kept (noise is dropped);
 *                  d_out_xyz NULL: no compaction (d_out_rgb and d_out_index NULL too)
 * eps finite and > 0 with eps * eps > 0; min_points >= 0; min_size >= 1. */
int d2pc_dbscan_enqueue(const float *d_xyz, const float *d_rgb, const uint32_t *d_count, uint32_t capacity_rows,
                        const float *d_bounds, double eps, int32_t min_points, uint32_t min_size, void *d_scratch,
                        size_t scratch_bytes, int32_t *d_out_labels, uint32_t *d_out_sizes, float *d_out_xyz,
                        float *d_out_rgb, uint32_t *d_out_index, uint32_t *d_out_counts, void *stream);

/* Point normals (Open3D PointCloud::EstimateNormals with fast_normal_computation, then
 * OrientNormalsTowardsCameraLocation) on ONE frame's rows, through the same grid as statistical outlier removal:
 * the knn nearest points (the point itself included, float64 distances, ties ordered by (d2, source row)); with
 * radius > 0 only points with d2 < radius^2 (Open3D's hybrid search); covariance of those neighbours (identity when
 * fewer than 3), eigenvector of its smallest eigenvalue (Geometric Tools' robust 3x3 solver, float64), normalised,
 * (0, 0, 1) when the covariance is zero; with orient != 0 flipped where n . (camera - p) < 0.
 *   d_bounds       float32 [6] min/max of the rows (emit want_bounds = 1, or d2pc_rows_bounds_enqueue)
 *   knn            1..64;  radius <= 0: k-NN mode (NaN is refused)
 *   camera         HOST pointer to 3 doubles, read during the call; may be NULL when orient == 0
 *   d_scratch      d2pc_normals_scratch_bytes(capacity_rows) bytes, 256-byte aligned
 *   d_out_normals  float64 [capacity_rows, 3], row i = normal of input row i
 *   d_out_cov      float64 [capacity_rows, 6] = c00, c01, c02, c11, c12, c22 of every row, or NULL
 * Argument errors are returned before any launch; the call does not synchronise. */
int d2pc_normals_scratch_bytes(uint32_t capacity_rows, size_t *bytes);
int d2pc_normals_enqueue(const float *d_xyz, const uint32_t *d_count, uint32_t capacity_rows,
                         const float *d_bounds, int32_t knn, double radius, int32_t orient,
                         const double camera[3], void *d_scratch, size_t scratch_bytes,
                         double *d_out_normals, double *d_out_cov, void *stream);

/* m1 -- triangle mesh of ONE frame's lattice: the rows of an unmasked emit (row i = r * cols + c of a rows x cols
 * lattice, i.e. ceil(H / step) x ceil(W / step)).  A row is a vertex candidate when d_keep[i] != 0 (or d_keep is
 * NULL) and its three coordinates are finite.  Quad (r, c) has corners a (r, c), b (r, c+1), p (r+1, c), d (r+1, c+1):
 * with four valid corners it is split along a-d into (a, p, d), (a, d, b) when d2(a, d) <= d2(b, p), else along b-p
 * into (a, p, b), (b, p, d); with three valid corners it gives the triangle of those three (in this winding).  A
 * triangle is kept when, in float64 with n = (p1 - p0) x (p2 - p0) and s = (p0 + p1) + p2: n.n > 0, n.s < 0 (it
 * faces the camera), (n.s)^2 >= cos2 (n.n)(s.s) (it is not grazing: depth discontinuities are dropped), and, with
 * max_edge > 0, every edge has d2 <= max_edge^2.
 *   flags          D2PC_MESH_REMOVE_UNREFERENCED: only rows used by a kept triangle become vertices (else every valid
 *                  row); D2PC_MESH_NORMALS: vertex normals (Open3D ComputeVertexNormals: the unnormalised n of the
 *                  adjacent kept triangles summed in ascending triangle order, normalised; (0, 0, 1) for a zero sum)
 *   cos2           cos(max_angle)^2 in [0, 1];  max_edge <= 0: no edge limit (NaN / inf are refused)
 *   d_scratch      d2pc_grid_mesh_scratch_bytes(rows, cols) bytes, 256-byte aligned
 *   d_vtx_xyz/rgb  float32 [rows * cols, 3]; d_vtx_row int32 [rows * cols] lattice row of every vertex;
 *                  d_vtx_normals float64 [rows * cols, 3] (needed with D2PC_MESH_NORMALS, else may be NULL);
 *                  d_vtx_count uint32 [1]; vertices in lattice order
 *   d_tri          int32 [2 (rows - 1)(cols - 1), 3] vertex ids (may be NULL when rows or cols is 1);
 *                  d_tri_count uint32 [1]; triangles ordered by quad, (a, p, *) first
 * rows * cols must be below 2^31.  Argument errors are returned before any launch; the call does not synchronise
 * and the result repeats bit for bit. */
enum { D2PC_MESH_REMOVE_UNREFERENCED = 1, D2PC_MESH_NORMALS = 2 };
int d2pc_grid_mesh_scratch_bytes(uint32_t rows, uint32_t cols, size_t *bytes);
int d2pc_grid_mesh_enqueue(const float *d_xyz, const float *d_rgb, const uint8_t *d_keep, uint32_t rows,
                           uint32_t cols, double max_edge, double cos2, uint32_t flags, void *d_scratch,
                           size_t scratch_bytes, float *d_vtx_xyz, float *d_vtx_rgb, int32_t *d_vtx_row,
                           double *d_vtx_normals, uint32_t *d_vtx_count, int32_t *d_tri, uint32_t *d_tri_count,
                           void *stream);

/* Binary little-endian PLY faces as Open3D's write_triangle_mesh writes them ("property list uchar uint
 * vertex_indices"), 13 bytes each: uchar 3, then three uint32 vertex ids.  d_tri int32 [capacity, 3] with
 * *d_tri_count <= capacity rows in use; d_records 16-byte aligned, capacity * 13 bytes. */
int d2pc_ply_face_records_enqueue(const int32_t *d_tri, const uint32_t *d_tri_count, uint32_t capacity,
                                  uint8_t *d_records, void *stream);

/* m2 -- simplification of ONE triangle mesh by vertex clustering (Open3D SimplifyVertexClustering; our own rules,
 * oracle/d2pc_simplify_oracle.py).  Vertices are binned with the ax-2 voxel rule (bmin = the vertices' minimum,
 * vmin = bmin - vs/2, idx = floor((v - vmin) / vs) in float64, idx < 2^21).  Every occupied cluster becomes one vertex,
 * ordered by its lowest member vertex id, whose vertex row it takes; its colour is the members' mean, its normal
 * (with D2PC_SIMPLIFY_NORMALS) the members' normalised sum ((0, 0, 0) for a zero sum), its position the members' mean
 * or, with D2PC_SIMPLIFY_QUADRIC, the minimiser x = -A^-1 b of the summed plane quadrics of the triangles at its
 * members (A = sum of area n n^T, b = sum of area d n, once per triangle corner) when det A > 1e-4 trace(A)^3 and x
 * lies in the cluster's own cell, else the mean.  Triangles are mapped to cluster ids; collapsed ones are dropped,
 * the rest rotated to start at their smallest id, and only the first of each rotation (by input index) stays, in
 * input order.
 *   d_vtx_xyz/rgb     float32 [vertices, 3]; d_vtx_normals float64 [vertices, 3] (with D2PC_SIMPLIFY_NORMALS);
 *                     d_vtx_row int64 [vertices]; d_tri int32 [triangles, 3]
 *   d_scratch         d2pc_mesh_simplify_scratch_bytes(vertices, triangles) bytes, 256-byte aligned
 *   d_out_xyz/rgb     float32 [vertices, 3]; d_out_normals float64 [vertices, 3] (with D2PC_SIMPLIFY_NORMALS);
 *                     d_out_row int64 [vertices]; d_out_vtx_count uint32 [1]
 *   d_out_tri         int32 [triangles, 3]; d_out_tri_count uint32 [1]
 *   d_error           int32 [1]: bit 1 = a cluster index >= 2^21 (voxel_size too small), bit 2 = a triangle id
 *                     outside [0, vertices), bit 4 = a vertex with a non-finite coordinate, colour or normal; any
 *                     error leaves both counts 0
 * Sums are 64-bit fixed point (positions and the quadric scaled to the mesh's extent and total area, colours to
 * their largest magnitude, normals in two words), so the result repeats bit for bit: colour means are exact for
 * integral colours, position means are within 2^-38 * extent of the exact means (plus the float32 rounding).
 * voxel_size finite and > 0; vertices >= 2^24 or triangles >= 2^31 return D2PC_ERR_UNSUPPORTED.  Argument errors
 * are returned before any launch; the call does not synchronise. */
enum { D2PC_SIMPLIFY_QUADRIC = 1, D2PC_SIMPLIFY_NORMALS = 2 };
int d2pc_mesh_simplify_scratch_bytes(uint32_t vertices, uint32_t triangles, size_t *bytes);
int d2pc_mesh_simplify_enqueue(const float *d_vtx_xyz, const float *d_vtx_rgb, const double *d_vtx_normals,
                               const int64_t *d_vtx_row, uint32_t vertices, const int32_t *d_tri, uint32_t triangles,
                               double voxel_size, uint32_t flags, void *d_scratch, size_t scratch_bytes,
                               float *d_out_xyz, float *d_out_rgb, double *d_out_normals, int64_t *d_out_row,
                               uint32_t *d_out_vtx_count, int32_t *d_out_tri, uint32_t *d_out_tri_count,
                               int32_t *d_error, void *stream);

/* m3 -- connected components of ONE triangle mesh (Open3D ClusterConnectedTriangles; our restatement,
 * oracle/d2pc_components_oracle.py).  Two triangles are connected when they share an edge, an unordered vertex pair
 * (sharing only a vertex does not connect; a non-manifold edge connects every triangle on it; a degenerate triangle
 * (a, a, b) has the edges {a,a}, {a,b}, {a,b}).  Clusters are numbered in ascending order of their lowest triangle.
 * The area of a triangle is Open3D's 0.5 |(p0 - p1) x (p0 - p2)| in float64 (Eigen's component order, the norm summed
 * left to right); the area of a cluster is sum_t rint(a_t s) / s in 64-bit fixed point with s = 2^(62 - e_a - e_T),
 * max_t a_t < 2^e_a (frexp; e_a = 0 when every area is 0) and T <= 2^e_T, the integer sum rounded once to float64.
 *   d_vtx_xyz            float32 [vertices, 3]; d_tri int32 [triangles, 3]
 *   d_scratch            d2pc_mesh_components_scratch_bytes(vertices, triangles) bytes, 256-byte aligned
 *   d_out_tri_cluster    int32 [triangles]: cluster of every triangle
 *   d_out_cluster_n      int64 [triangles], the first K in use: triangles of every cluster
 *   d_out_cluster_area   float64 [triangles], the first K in use: area of every cluster
 *   d_out_cluster_count  uint32 [1]: K (0 on an error)
 *   d_error              int32 [1]: bit 1 = a triangle id outside [0, vertices), bit 2 = a vertex with a non-finite
 *                        coordinate, bit 4 = a loop bound was exhausted (an internal failure, never expected)
 * triangles <= 2^25 (twice the 2 * 2159 * 3839 triangles of a 4K lattice mesh) and vertices <= 2^31, else
 * D2PC_ERR_UNSUPPORTED.  No floating-point atomics: the result repeats bit for bit.  Argument errors are returned
 * before any launch; the call does not synchronise. */
int d2pc_mesh_components_scratch_bytes(uint32_t vertices, uint32_t triangles, size_t *bytes);
int d2pc_mesh_components_enqueue(const float *d_vtx_xyz, uint32_t vertices, const int32_t *d_tri, uint32_t triangles,
                                 void *d_scratch, size_t scratch_bytes, int32_t *d_out_tri_cluster,
                                 int64_t *d_out_cluster_n, double *d_out_cluster_area, uint32_t *d_out_cluster_count,
                                 int32_t *d_error, void *stream);

/* m3 -- removal of triangles by a mask (Open3D RemoveTrianglesByMask, then with D2PC_MESH_REMOVE_UNREFERENCED
 * RemoveUnreferencedVertices).  Triangle t stays when d_tri_keep[t] != 0; kept triangles keep their input order.
 * Vertices stay in input order (with D2PC_MESH_REMOVE_UNREFERENCED only those a kept triangle uses), their colour,
 * row and (with D2PC_MESH_NORMALS) normal carried unchanged, and the kept triangles are remapped to the new ids.
 *   d_vtx_xyz/rgb        float32 [vertices, 3]; d_vtx_normals float64 [vertices, 3] (with D2PC_MESH_NORMALS);
 *                        d_vtx_row int64 [vertices]; d_tri int32 [triangles, 3]; d_tri_keep uint8 [triangles]
 *   d_scratch            d2pc_mesh_filter_scratch_bytes(vertices, triangles) bytes, 256-byte aligned
 *   d_out_xyz/rgb        float32 [vertices, 3]; d_out_normals float64 [vertices, 3] (with D2PC_MESH_NORMALS);
 *                        d_out_row int64 [vertices]; d_out_vtx_count uint32 [1]
 *   d_out_tri            int32 [triangles, 3]; d_out_tri_count uint32 [1]
 *   d_error              int32 [1]: bit 1 = a triangle id outside [0, vertices), bit 2 = a vertex with a non-finite
 *                        coordinate; any error leaves both counts 0
 * The size limits are those of d2pc_mesh_components_enqueue.  Argument errors are returned before any launch; the
 * call does not synchronise. */
int d2pc_mesh_filter_scratch_bytes(uint32_t vertices, uint32_t triangles, size_t *bytes);
int d2pc_mesh_filter_enqueue(const float *d_vtx_xyz, const float *d_vtx_rgb, const double *d_vtx_normals,
                             const int64_t *d_vtx_row, uint32_t vertices, const int32_t *d_tri, uint32_t triangles,
                             const uint8_t *d_tri_keep, uint32_t flags, void *d_scratch, size_t scratch_bytes,
                             float *d_out_xyz, float *d_out_rgb, double *d_out_normals, int64_t *d_out_row,
                             uint32_t *d_out_vtx_count, int32_t *d_out_tri, uint32_t *d_out_tri_count,
                             int32_t *d_error, void *stream);

/* m4 -- smoothing of ONE triangle mesh (Open3D FilterSmoothSimple / FilterSmoothLaplacian / FilterSmoothTaubin; our
 * restatement, oracle/d2pc_smooth_oracle.py).  The neighbours of a vertex are Open3D's adjacency sets (triangle
 * (a, b, c) adds b, c to adj[a], a, c to adj[b], a, b to adj[c]), visited in ascending vertex id.  The float32 input
 * is widened to float64, every pass reads the previous state (Jacobi) and the result is rounded to float32 once.
 *   SIMPLE      p' = (p + sum_nb p_nb) / (1 + |adj|)
 *   LAPLACIAN   w = 1 / (sqrt((dx dx + dy dy) + dz dz) + 1e-12) of p - p_nb, p' = p + lambda (sum w p_nb / sum w - p);
 *               a vertex without neighbours stays as it is
 *   TAUBIN      every iteration a LAPLACIAN pass with lambda_filter, then one with mu
 * Every sum runs left to right from zero.  `scope` is a non-empty set of D2PC_SMOOTH_VERTEX / _NORMAL / _COLOR
 * (Open3D's FilterScope); colours and normals take the positions' weights; normals are filtered only when given and
 * are not renormalised; the other fields are copied.  0 iterations copy everything.
 *   d_vtx_xyz/rgb     float32 [vertices, 3]; d_vtx_normals float64 [vertices, 3] or NULL; d_tri int32 [triangles, 3]
 *   d_scratch         d2pc_mesh_smooth_scratch_bytes(vertices, triangles) bytes, 256-byte aligned
 *   d_out_xyz/rgb     float32 [vertices, 3]; d_out_normals float64 [vertices, 3] (NULL exactly when d_vtx_normals
 *                     is); outputs must not overlap the inputs
 *   d_error           int32 [1]: bit 1 = a triangle id outside [0, vertices), bit 2 = a non-finite coordinate (or
 *                     colour / normal in the scope), bit 4 = a loop bound was exhausted (an internal failure, never
 *                     expected); any error leaves the filtered outputs undefined
 * triangles <= 2^25 and vertices <= 2^31, else D2PC_ERR_UNSUPPORTED.  lambda_filter and mu finite; an unknown method
 * or scope and every other argument error are returned before any launch.  No floating-point atomics: the result
 * repeats bit for bit.  The call does not synchronise. */
enum { D2PC_SMOOTH_SIMPLE = 0, D2PC_SMOOTH_LAPLACIAN = 1, D2PC_SMOOTH_TAUBIN = 2 };
enum { D2PC_SMOOTH_VERTEX = 1, D2PC_SMOOTH_NORMAL = 2, D2PC_SMOOTH_COLOR = 4 };
int d2pc_mesh_smooth_scratch_bytes(uint32_t vertices, uint32_t triangles, size_t *bytes);
int d2pc_mesh_smooth_enqueue(const float *d_vtx_xyz, const float *d_vtx_rgb, const double *d_vtx_normals,
                             uint32_t vertices, const int32_t *d_tri, uint32_t triangles, int method,
                             uint32_t iterations, double lambda_filter, double mu, uint32_t scope,
                             void *d_scratch, size_t scratch_bytes, float *d_out_xyz, float *d_out_rgb,
                             double *d_out_normals, int32_t *d_error, void *stream);

/* m4 -- vertex normals of ANY triangle mesh, m1's rule (Open3D ComputeVertexNormals): the unnormalised
 * (p1 - p0) x (p2 - p0) of every triangle in float64, summed per vertex in ascending triangle order once per corner,
 * then v / sqrt(v.v), (0, 0, 1) for a zero sum.  Equals d2pc_grid_mesh_enqueue's normals bit for bit.
 *   d_vtx_xyz float32 [vertices, 3]; d_tri int32 [triangles, 3]; d_out_normals float64 [vertices, 3]
 *   d_scratch d2pc_mesh_vertex_normals_scratch_bytes(vertices, triangles) bytes, 256-byte aligned
 *   d_error   as d2pc_mesh_smooth_enqueue's (bit 2: a non-finite coordinate)
 * The size limits are those of d2pc_mesh_smooth_enqueue.  Argument errors are returned before any launch; the call
 * does not synchronise. */
int d2pc_mesh_vertex_normals_scratch_bytes(uint32_t vertices, uint32_t triangles, size_t *bytes);
int d2pc_mesh_vertex_normals_enqueue(const float *d_vtx_xyz, uint32_t vertices, const int32_t *d_tri,
                                     uint32_t triangles, void *d_scratch, size_t scratch_bytes,
                                     double *d_out_normals, int32_t *d_error, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* D2PC_H_ */
