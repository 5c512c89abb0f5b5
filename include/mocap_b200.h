/* mocap_b200.h -- C-ABI of the B200-native MocapV2 capture hot path (libmocap_b200.so, sm_100a).
 *
 * The reference (RashmikaDushan/MocapV2) has no FFI: its "operator interface" for this path is the set of
 * module-level Python functions in lib/ImageOperations.py and lib/Helpers.py.  Each entry point below is
 * what a ctypes binding of one of those functions binds (see INTEGRATION.md for the stub); the reference
 * interface it replaces is cited as file:line of /root/reference.
 *
 * Conventions: every *_dev pointer is device memory owned by the caller (torch tensors in the Python host
 * layer); `stream` is a cudaStream_t passed as void*; all calls are asynchronous on that stream, allocate
 * nothing, keep no global state and are re-entrant.  Everything a call reads is in its arguments: a handle (stage timer, detection
 * pipe) owns CUDA streams and events and remembers what its last call ran, nothing more.  Return value: MOCAP_OK or a negative
 * status; per-frame / per-frame-set problems (capacity overflows) are reported in the flags arrays, not in the return value.
 */
#ifndef MOCAP_B200_H
#define MOCAP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MOCAP_OK 0
#define MOCAP_ERR_INVALID (-1)     /* bad argument (null pointer, non-positive size, unsupported shape) */
#define MOCAP_ERR_WORKSPACE (-2)   /* workspace smaller than mocap_*_workspace_bytes() */
#define MOCAP_ERR_CUDA (-3)        /* a CUDA runtime call failed (cudaGetLastError() is preserved) */
#define MOCAP_ERR_UNSUPPORTED (-4) /* shape outside the compiled limits (frame side > 16384, > MOCAP_MAX_CAMS views, displacement > 1023 px) */

/* per-frame flags written to out_flags[] of mocap_detect_batch */
#define MOCAP_FLAG_RUN_OVERFLOW 1      /* more foreground runs than max_runs: frame outputs invalid */
#define MOCAP_FLAG_BLOB_OVERFLOW 2     /* more kept centroids than max_blobs: list truncated */
#define MOCAP_FLAG_CONTOUR_OVERFLOW 4  /* more contours than max_contours: frame outputs invalid */
#define MOCAP_FLAG_TILE_OVERFLOW 8     /* more foreground tiles than the workspace holds */
#define MOCAP_FLAG_DEPTH_OVERFLOW 16   /* contour tree deeper than 8: order resolved by the slow path */
#define MOCAP_FLAG_TRACE_OVERFLOW 32   /* a border longer than the step budget: frame outputs invalid */
#define MOCAP_FLAG_GENERAL_PATH 64     /* informational: the frame was finished by the general per-frame path (hole borders,
                                          oversized blob groups, parity outputs requested), not by the per-cluster units; bits 8.. say why:
                                          2 too many hot cells, 3 too many clusters, 5 cluster storage full, 7 too many border
                                          starts, 8 border trace / hole parent outside the fast rules, 9 nested outer border,
                                          10 lens displacement varies by more than 8 px inside a 32-px cell */
#define MOCAP_FLAG_LENS_INDEX 128      /* the frame's lens index (MocapLensSet::frame_lens_dev) lies outside [0, n_lenses): count 0,
                                          no table was read for the frame */

/* per-frame-set flags written by mocap_correspond_batch */
#define MOCAP_CFLAG_GROUP_CAP 1        /* a root had more candidate groups than max_groups: mean over the first max_groups */
#define MOCAP_CFLAG_CAND_CAP 2         /* a (root, camera) pair had more in-cutoff candidates than MOCAP_MAX_CAND */
#define MOCAP_CFLAG_TIE 4              /* a distance within 1e-5 of the cutoff (Helpers.py:219), logged as a tie */

#define MOCAP_MAX_CAND 8               /* candidates kept per (root, camera), ascending distance */
#define MOCAP_MAX_CAMS 16              /* views per triangulation / cameras per frame-set */
#define MOCAP_CAM_STRIDE 40            /* doubles per camera record, see mocap_pack_camera layout below */

/* Camera record layout (doubles): [0..11] P = K[R|t] row-major 3x4 (Helpers.py:58-62)
 *                                 [12..20] R row-major, [21..23] t, [24..32] K row-major, [33..37] k1 k2 p1 p2 k3 */

const char* mocap_status_string(int status);
int mocap_abi_version(void);
/* kernels launched by this library in this process so far (every launch is counted where it is issued) */
unsigned long long mocap_kernel_launch_count(void);

/* ---- undistortion table: cv.undistort(img, K0, dist0) of _find_dot (lib/ImageOperations.py:37-38) -------
 * Built once per (K, dist, H, W).  Holds the 1/32-px fixed-point displacement map of
 * cv::initUndistortRectifyMap (FP64, same operation order) plus the source-cell -> output-tile reach table. */
size_t mocap_undistort_table_bytes(int H, int W);
int mocap_undistort_table_build(const double* K9_host, const double* dist5_host, int H, int W,
                                void* table_dev, size_t table_bytes, void* stream);

/* ---- detection: _find_dot(img)[1] for a batch of frames (lib/ImageOperations.py:33-78) --------------------
 * frames_dev: n_frames x H x W uint8 (row stride W, frame stride `frame_stride` bytes).
 * out_xy[n][max_blobs][2] int32 centroids in the reference's output order, out_count[n] how many
 * (0 = the reference's [[None, None]]), out_flags[n] MOCAP_FLAG_*.
 * Centroid of a kept contour: q = (m10 / m00, m01 / m00), the FP64 quotients of cv.moments of the contour polygon (lib/ImageOperations.py:
 * 59-62).  The entry points without a suffix store int(q) (truncated toward zero, the reference's whole pixels); the *_subpixel entry
 * points store (float)q, the float32 nearest to q (spacing <= 2^-10 px below 16384), in the same 8-byte slot: out_xy[n][max_blobs][2]
 * float32.  Contours, filter, order, counts and flags do not depend on the format.
 * Optional (may be NULL) parity outputs:
 *   out_bits[n][H][ceil(W/32)]   the filtered binary image (image_filter_gpu, :23-31), LSB = leftmost pixel
 *   out_labels[n][H][W] int32    8-connected blob labels, 0 = background, k = k-th blob in raster order
 *   out_blob_sums[n][max_blobs][3] int64  per-blob pixel m00, m10, m01;  out_blob_count[n]
 *   out_contours[n][max_contours][8] double: a00, a10, a01 (exact integers), perimeter, is_hole,
 *                                   parent (index in output order or -1), kept, start pixel index
 *   out_contour_count[n]
 * Workspace: mocap_detect_workspace_bytes(), sized for the parity outputs.  The overlapped call below uses the same layout with one
 * cluster-path block per chunk instead of one for the batch.
 */
size_t mocap_detect_workspace_bytes(int n_frames, int H, int W, int max_blobs, int max_contours, int max_runs);

/* ---- lens set: one undistortion table per camera ------------------------------------------------------------------------
 * n_lenses tables of one frame size, each built by mocap_undistort_table_build, lens l at tables_dev + l * lens_stride (one device
 * allocation).  frame_lens_dev [n_frames] int32: the lens of every frame of a call (device memory, complete on the call's stream);
 * NULL = lens 0 for every frame.  A frame whose index lies outside [0, n_lenses) gets count 0 and MOCAP_FLAG_LENS_INDEX.
 * One table is the set {table_dev, 1, mocap_undistort_table_bytes(H, W), NULL}.  A call reads the structure before it returns; the
 * device arrays must stay valid until its kernels have run.  MOCAP_ERR_INVALID: a NULL set or tables_dev, n_lenses < 1,
 * lens_stride < mocap_undistort_table_bytes(H, W) or not a multiple of 256. */
typedef struct MocapLensSet {
    const void* tables_dev;
    int n_lenses;
    size_t lens_stride;
    const int32_t* frame_lens_dev;
} MocapLensSet;

/* Optional per-stage device timing of mocap_detect_batch (bench.py's roofline line): a timer owns CUDA events that
 * the call records around its kernels on `stream`; read it after the stream has been synchronised.  Stages:
 * 0 scan (streams every source byte), 1 group (hot cells -> clusters -> 64x64 filter pieces), 2 filter (remap + floor-mean
 * threshold + majority per piece, in shared memory), 3 borders (per frame: border-start candidates, Suzuki-Abe traces,
 * filter / centroid / order), 4 finish (general path for the frames that need it).  ms_out[MOCAP_N_STAGES], -1 for a
 * stage that was not recorded. */
#define MOCAP_N_STAGES 5
void* mocap_stage_timer_create(void);
void mocap_stage_timer_destroy(void* timer);
int mocap_stage_timer_read(void* timer, float* ms_out);
const char* mocap_stage_name(int stage);
int mocap_detect_batch(const uint8_t* frames_dev, int n_frames, int H, int W, int64_t frame_stride,
                       const MocapLensSet* lenses, int thresh, double min_area, double min_circ,
                       int max_blobs, int max_contours, int max_runs,
                       int32_t* out_xy, int32_t* out_count, int32_t* out_flags,
                       uint32_t* out_bits, int32_t* out_labels, int64_t* out_blob_sums, int32_t* out_blob_count,
                       double* out_contours, int32_t* out_contour_count,
                       void* workspace, size_t workspace_bytes, void* stream, void* stage_timer_or_null);
/* The same with sub-pixel centroids: out_xy [n][max_blobs][2] float32 (see the centroid definition above). */
int mocap_detect_batch_subpixel(const uint8_t* frames_dev, int n_frames, int H, int W, int64_t frame_stride,
                                const MocapLensSet* lenses, int thresh, double min_area, double min_circ,
                                int max_blobs, int max_contours, int max_runs,
                                float* out_xy, int32_t* out_count, int32_t* out_flags,
                                uint32_t* out_bits, int32_t* out_labels, int64_t* out_blob_sums, int32_t* out_blob_count,
                                double* out_contours, int32_t* out_contour_count,
                                void* workspace, size_t workspace_bytes, void* stream, void* stage_timer_or_null);

/* ---- overlapped detection (same results as mocap_detect_batch without the parity outputs) ----------------------------
 * The batch is cut into chunks of `chunk_frames` frames (<= 0: one chunk); chunk k's stages (group, piece filter, borders) run as
 * one chain on worker stream k mod n_worker_streams of the pipe.  The streaming scan -- one TMA-fed kernel (cp.async.bulk.tensor +
 * mbarrier ring in shared memory, one small CTA per SM) over the whole batch on the pipe's high-priority scan stream -- runs
 * beside the stages of the chunks it has already finished, which wait for its per-chunk flag with a stream memory operation.
 * Frames the TMA unit cannot describe (rows or frame stride not a multiple of 16 bytes, thresh outside 0..254), or a driver
 * without stream memory operations, take the classic scan kernels chunk by chunk, handed over with events; with cell boxes handed in
 * there is no scan.  A pipe owns those streams and events and remembers what its last call ran: create one per caller thread, keep it
 * for the life of the engine; a call is asynchronous on `stream` like every other entry point (fork / join with events).
 * record_timeline != 0 keeps the call's timeline for mocap_detect_pipe_timeline.  Frame sizes the per-cluster units do not support
 * return MOCAP_ERR_UNSUPPORTED (use mocap_detect_batch).
 * Optional inputs of a call (NULL: not used):
 *   cellbox_dev [n_frames][ceil(H/32)][ceil(W/32)]: the frames' hot cell boxes, complete on `stream` before the call, as written by
 *     mocap_scan_cells_batch or mocap_bayer_gr2gray_scan_batch for the same frames and thresh.  The call then runs no streaming scan.
 *   xy_dst_dev, count_dst_dev [n_frames] device addresses (both or neither; one without the other is MOCAP_ERR_INVALID): the
 *     store-to-peer epilogue (multi-GPU).  Every frame's record is ALSO copied -- chunk by chunk, behind the chunk's border stage --
 *     to xy_dst[f] (its centroids, int32 pairs; float32 pairs in the _subpixel call) and count_dst[f] (its count): addresses in the receive buffer of the rank that
 *     matches the frame's frame-set, mapped into this process (symmetric memory over NVLink).  The exchange step is then a barrier.
 *   scan_wait_event, scan_done_event (cudaEvent_t owned by the caller): the scan token of several pipes in flight on one GPU
 *     (pipeline.StepsInFlight).  The call's streaming scan waits for scan_wait_event and records scan_done_event behind it.
 *     Chained from call to call across the pipes, the HBM-bound scans run one after the other instead of side by side: one ring
 *     of TMA boxes per SM instead of two. */
void* mocap_detect_pipe_create(int n_worker_streams);
void mocap_detect_pipe_destroy(void* pipe);
/* the workspace layout of mocap_detect_workspace_bytes with the call's chunk count (chunk_frames as in the call) */
size_t mocap_detect_pipelined_workspace_bytes(int n_frames, int H, int W, int max_blobs, int max_contours, int max_runs, int chunk_frames);
int mocap_detect_batch_pipelined(void* pipe, const uint8_t* frames_dev, int n_frames, int H, int W, int64_t frame_stride,
                                 const MocapLensSet* lenses, int thresh, double min_area, double min_circ,
                                 int max_blobs, int max_contours, int max_runs,
                                 int32_t* out_xy, int32_t* out_count, int32_t* out_flags,
                                 double* out_contours, int32_t* out_contour_count,
                                 const uint32_t* cellbox_dev, const uint64_t* xy_dst_dev, const uint64_t* count_dst_dev,
                                 void* scan_wait_event, void* scan_done_event,
                                 void* workspace, size_t workspace_bytes, void* stream, int chunk_frames, int record_timeline);
/* The same with sub-pixel centroids: out_xy [n][max_blobs][2] float32, and xy_dst[f] receives float32 pairs. */
int mocap_detect_batch_pipelined_subpixel(void* pipe, const uint8_t* frames_dev, int n_frames, int H, int W, int64_t frame_stride,
                                          const MocapLensSet* lenses, int thresh, double min_area, double min_circ,
                                          int max_blobs, int max_contours, int max_runs,
                                          float* out_xy, int32_t* out_count, int32_t* out_flags,
                                          double* out_contours, int32_t* out_contour_count,
                                          const uint32_t* cellbox_dev, const uint64_t* xy_dst_dev, const uint64_t* count_dst_dev,
                                          void* scan_wait_event, void* scan_done_event,
                                          void* workspace, size_t workspace_bytes, void* stream, int chunk_frames, int record_timeline);
/* ms since the fork of the last call with record_timeline: [scan done, join] then per chunk [scan seen, grouped, filtered,
 * borders done]; returns the number of floats written, 0 without a timeline */
int mocap_detect_pipe_timeline(void* pipe, float* ms_out, int cap);
/* what the last call ran: out2 = {scan kernel (1 TMA ring: the workers waited on its chunk flags; 0 classic scan or none), chunks} */
int mocap_detect_pipe_info(void* pipe, int* out2);

/* stage entry points of the same path (used by the parity tests and the bench's per-kernel timing) */
/* the streaming scan alone: cellbox_out [n][ceil(H/32)][ceil(W/32)] hot bounding box of every 32x32 source cell
 * (x0 | x1 << 8 | y0 << 16 | y1 << 24, 0xffffffff: no pixel > thresh).  variant 0 classic kernels, 1 TMA ring (workspace >= 1 KB);
 * any other variant returns MOCAP_ERR_INVALID */
int mocap_scan_cells_batch(const uint8_t* frames_dev, int n_frames, int H, int W, int64_t frame_stride, const void* table_dev,
                           int thresh, int variant, uint32_t* cellbox_out, void* workspace, size_t workspace_bytes, void* stream);
int mocap_filter_batch(const uint8_t* frames_dev, int n_frames, int H, int W, int64_t frame_stride,
                       const void* table_dev, int thresh, uint32_t* out_bits,
                       void* workspace, size_t workspace_bytes, void* stream);

/* cv.findContours(RETR_TREE, CHAIN_APPROX_SIMPLE) -> area/circularity filter -> cv.moments centroid on a given packed
 * binary image bits_dev [n][H][ceil(W/32)] (lib/ImageOperations.py:41-65); bits at x >= W must be zero.  Outputs as in
 * mocap_detect_batch; workspace of mocap_detect_workspace_bytes(). */
int mocap_blobs_batch(const uint32_t* bits_dev, int n_frames, int H, int W,
                      double min_area, double min_circ, int max_blobs, int max_contours, int max_runs,
                      int32_t* out_xy, int32_t* out_count, int32_t* out_flags,
                      int32_t* out_labels, int64_t* out_blob_sums, int32_t* out_blob_count,
                      double* out_contours, int32_t* out_contour_count,
                      void* workspace, size_t workspace_bytes, void* stream);

/* cv.drawContours(img, contours_filtered, -1, (0,0,255), 2) of _find_dot (lib/ImageOperations.py:52-55; display only): paints `value`
 * (the reference's colour on a one-channel image: 0) over the thickness-2 outline of every KEPT contour of the table returned by
 * mocap_detect_batch (out_contours / out_contour_count, with the packed binary image out_bits of the same call) into img_dev [n][H][W].
 * H, W <= 16384 as for mocap_detect_batch. */
int mocap_draw_contours_batch(const uint32_t* bits_dev, const double* contours_dev, const int32_t* contour_count_dev,
                              int n_frames, int H, int W, int max_contours, uint8_t* img_dev, int value, void* stream);

/* ---- the reference's own GPU op: fast_cuda_blur(image, 5) (lib/CudaOperations.py:24-41) -------------------- */
int mocap_blur5_batch(const uint8_t* frames_dev, int n_frames, int H, int W, uint8_t* out_dev, void* stream);
/* image_filter_cpu (lib/ImageOperations.py:15-21): cv.medianBlur(image, 5) then cv.threshold(., thresh, 255, BINARY) -> u8 {0,255} */
int mocap_median5_threshold_batch(const uint8_t* frames_dev, int n_frames, int H, int W, int thresh, uint8_t* out_dev, void* stream);
/* Bayer front step of the realtime loop: cv2.cvtColor(raw, COLOR_BAYER_GR2BGR) then cv2.cvtColor(., COLOR_BGR2GRAY)
 * (RealtimeTracking_FLIR.py:103-104), fused: raw u8 [n][H][W] -> grey u8 [n][H][W].  H, W >= 3. */
int mocap_bayer_gr2gray_batch(const uint8_t* raw_dev, int n_frames, int H, int W, uint8_t* out_dev, void* stream);
/* The same front step, which also delivers what the streaming scan of the detection would compute from the grey frames it writes:
 * cellbox_out [n][ceil(H/32)][ceil(W/32)] as mocap_scan_cells_batch (the grey bytes are tested while they are in registers).  Passed as
 * cellbox_dev of mocap_detect_batch_pipelined, the detection of raw sensor frames (RealtimeTracking_FLIR.py:103-105) reads every frame
 * byte once less.  workspace >= n * ceil(H/32) * ceil(W/32) * 8 bytes. */
int mocap_bayer_gr2gray_scan_batch(const uint8_t* raw_dev, int n_frames, int H, int W, uint8_t* out_dev, int thresh,
                                   uint32_t* cellbox_out, void* workspace, size_t workspace_bytes, void* stream);
/* cv.undistort alone (lib/ImageOperations.py:38), for stage parity */
int mocap_undistort_batch(const uint8_t* frames_dev, int n_frames, int H, int W, const void* table_dev,
                          uint8_t* out_dev, void* stream);

/* ---- triangulation + reprojection error: triangulate_points / calculate_reprojection_errors ----------------
 * (lib/Helpers.py:43-99 DLT on B = A^T A, smallest singular vector; :102-143 mean squared pixel residual
 * through cv.projectPoints incl. distortion and its float32 roundings.)
 * pts_dev [P][C][2]: float32 (fp64_mode 0) or float64 (fp64_mode 1).  valid_dev [P][C] uint8 or NULL (all valid).
 * xyz_out [P][3], err_out [P] in the same dtype as pts; points with fewer than 2 valid views get NaN
 * (the reference's [None, None, None], Helpers.py:55-56).  err_out may be NULL. */
int mocap_triangulate_batch(const void* pts_dev, const uint8_t* valid_dev, const double* cams_dev, int C,
                            int64_t P, int fp64_mode, void* xyz_out, void* err_out, void* stream);
/* reprojection error of given object points (Helpers.py:102-143), same dtypes as above */
int mocap_reproject_batch(const void* pts_dev, const uint8_t* valid_dev, const void* xyz_dev,
                          const double* cams_dev, int C, int64_t P, int fp64_mode, void* err_out, void* stream);

/* The residual of bundle_adjustment (lib/Helpers.py:158-176; residual :160-167 = triangulate_points + calculate_reprojection_errors on
 * all points) under n_sets pose hypotheses in one launch, FP64: cams_sets_dev [n_sets][C][MOCAP_CAM_STRIDE], pts_dev [P][C][2] (every view
 * valid), err_out [n_sets][P].  One call per optimiser iteration evaluates the residual at x and at every x + h e_i of scipy's 2-point
 * finite-difference Jacobian. */
int mocap_ba_residuals_batch(const double* pts_dev, const double* cams_sets_dev, int n_sets, int C, int64_t P,
                             double* err_out, void* stream);

/* ---- epipolar correspondence + candidate groups + ranking ---------------------------------------------------
 * find_point_correspondance_and_object_points (lib/Helpers.py:178-280) for S frame-sets.
 * xy_dev [S][C][max_pts][2] int32 centroid lists (the [None, None] entry already dropped), count_dev [S][C].
 * F_dev [C-1][9]: Fs[i-1] maps camera-0 points to epilines in camera i (Helpers.py:205-207).
 * Outputs per frame-set: obj_out [S][max_pts][3] float64 object points sorted by mean reprojection error and
 * cut to obj_count+1 (Helpers.py:274-279) with n_obj_out[S]; img_out [S][max_pts][C][2] the first (all-closest)
 * group of every complete root in root order with n_valid_out[S]; err_out [S][max_pts] mean error per complete
 * root (root order); cand_out [S][max_pts][C][MOCAP_MAX_CAND] int32 candidate indices (-1 padded) or NULL;
 * flags_out [S] MOCAP_CFLAG_*. */
size_t mocap_correspond_workspace_bytes(int S, int C, int max_pts, int max_groups);
int mocap_correspond_batch(const int32_t* xy_dev, const int32_t* count_dev, int S, int C, int max_pts,
                           const double* F_dev, const double* cams_dev, double cutoff, int obj_count,
                           int max_groups, int fp64_mode,
                           double* obj_out, int32_t* n_obj_out, int32_t* img_out, int32_t* n_valid_out,
                           double* err_out, int32_t* cand_out, int32_t* flags_out,
                           void* workspace, size_t workspace_bytes, void* stream);

/* The same on centroid lists stored in camera blocks: xy_dev [C / cams_per_block][S][cams_per_block][max_pts][2], count_dev
 * [C / cams_per_block][S][cams_per_block] -- the buffer a rank holds after the shard exchange of the multi-GPU pipeline (one block per
 * source rank: that rank's cameras, this rank's frame-sets), read in place.  cams_per_block == C is mocap_correspond_batch. */
int mocap_correspond_batch_blocked(const int32_t* xy_dev, const int32_t* count_dev, int S, int C, int max_pts, int cams_per_block,
                                   const double* F_dev, const double* cams_dev, double cutoff, int obj_count,
                                   int max_groups, int fp64_mode,
                                   double* obj_out, int32_t* n_obj_out, int32_t* img_out, int32_t* n_valid_out,
                                   double* err_out, int32_t* cand_out, int32_t* flags_out,
                                   void* workspace, size_t workspace_bytes, void* stream);

/* mocap_correspond_batch_blocked on sub-pixel centroid lists (mocap_detect_batch_subpixel): xy_dev float32 and img_out
 * [S][max_pts][C][2] float32, everything else as there.  The roots' epilines are computed from the float32 points as the reference
 * does (Helpers.py:205-208), the distances and the DLT read them exactly. */
int mocap_correspond_batch_subpixel(const float* xy_dev, const int32_t* count_dev, int S, int C, int max_pts, int cams_per_block,
                                    const double* F_dev, const double* cams_dev, double cutoff, int obj_count,
                                    int max_groups, int fp64_mode,
                                    double* obj_out, int32_t* n_obj_out, float* img_out, int32_t* n_valid_out,
                                    double* err_out, int32_t* cand_out, int32_t* flags_out,
                                    void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MOCAP_B200_H */
