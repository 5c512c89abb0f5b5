// C-ABI glue of the detection path: workspace carving and the mocap_detect_batch / mocap_filter_batch entry points
// (include/mocap_b200.h).  _find_dot of the reference (lib/ImageOperations.py:33-78) = launch_filter + launch_blobs.
#include "common.cuh"
#include <string.h>

// detect_filter.cu
int table_view(const void* table_dev, int H, int W, TableView* tv);
int launch_scan(const uint8_t* frames, int n, int H, int W, int64_t fstride, const TableView& tv, int thresh,
                const FilterWs& ws, cudaStream_t s, StageTimer* timer);
int launch_tiles(const uint8_t* frames, int n, int H, int W, int64_t fstride, const TableView& tv, int thresh,
                 const FilterWs& ws, int max_fg, int* flags, const int* need_general, cudaStream_t s);
// detect_cluster.cu
size_t cluster_ws_bytes(int n, int H, int W, int max_contours, ClusterLayout* L);
bool cluster_path_supported(int H, int W);
int launch_cluster_path(const uint8_t* frames, int n, int H, int W, int64_t fstride, const TableView& tv, int thresh,
                        const uint32_t* cellbox, char* ws_base, const ClusterLayout& L, int* need_general,
                        int max_contours, int max_blobs, double min_area, double min_circ,
                        int32_t* out_xy, int xy_float, int32_t* out_count, int32_t* out_flags, double* out_contours, int32_t* out_contour_count,
                        cudaStream_t s, StageTimer* timer, const ClusterLaunch& how);
int launch_materialize_bits(const FilterWs& ws, int n, int H, int W, const TableView& tv, uint32_t* out, cudaStream_t s);
// detect_scan_tma.cu
bool scan_tma_supported(const uint8_t* frames, int n, int H, int W, int64_t fstride, int thresh);
size_t scan_tma_ctrl_bytes(int chunks);
const int* scan_tma_chunk_flag(const int* ctrl, int chunks, int chunk);
int launch_scan_tma(const uint8_t* frames, int n, int H, int W, int64_t fstride, const TableView& tv, int thresh, uint32_t* cellbox,
                    int* ctrl, int chunks, int chunk_frames, cudaStream_t s);
int stream_wait_geq(cudaStream_t s, const int* addr_dev, int value);
bool stream_wait_supported();
// detect_blobs.cu
int launch_tiles_from_bits(const uint32_t* bits, int n, int H, int TX, int TY, uint32_t* fg_tiles, int* n_fg, int max_fg, cudaStream_t s);
size_t blob_ws_stride(int H, int max_runs, int max_contours);
int launch_blobs(const uint32_t* bits, const uint32_t* fg_tiles, const int* n_fg, int n, int H, int W, int TX,
                 int max_fg, int max_runs, int max_blobs, int max_contours, double min_area, double min_circ,
                 char* ws, size_t ws_stride,
                 int32_t* out_xy, int xy_float, int32_t* out_count, int32_t* out_flags,
                 int64_t* out_blob_sums, int32_t* out_blob_count, double* out_contours, int32_t* out_contour_count,
                 int32_t* out_labels, const int* need_general, cudaStream_t s);

extern "C" const char* mocap_status_string(int status)
{
    switch (status) {
        case MOCAP_OK: return "ok";
        case MOCAP_ERR_INVALID: return "invalid argument";
        case MOCAP_ERR_WORKSPACE: return "workspace too small";
        case MOCAP_ERR_CUDA: return "CUDA runtime error";
        case MOCAP_ERR_UNSUPPORTED: return "shape outside the supported limits";
        default: return "unknown status";
    }
}

extern "C" int mocap_abi_version(void) { return MOCAP_ABI_VERSION; }

unsigned long long g_mocap_launches = 0;
extern "C" unsigned long long mocap_kernel_launch_count(void) { return __atomic_load_n(&g_mocap_launches, __ATOMIC_RELAXED); }

extern "C" const char* mocap_stage_name(int stage)
{
    static const char* names[MOCAP_N_STAGES] = {"scan", "group", "filter", "borders", "finish"};
    return (stage >= 0 && stage < MOCAP_N_STAGES) ? names[stage] : "?";
}

extern "C" void* mocap_stage_timer_create(void)
{
    StageTimer* t = new StageTimer();
    for (int i = 0; i < 2 * MOCAP_N_STAGES; ++i)
        if (cudaEventCreate(&t->ev[i]) != cudaSuccess) { delete t; return nullptr; }
    for (int i = 0; i < MOCAP_N_STAGES; ++i) t->recorded[i] = 0;
    return t;
}

extern "C" void mocap_stage_timer_destroy(void* timer)
{
    StageTimer* t = (StageTimer*)timer;
    if (!t) return;
    for (int i = 0; i < 2 * MOCAP_N_STAGES; ++i) cudaEventDestroy(t->ev[i]);
    delete t;
}

extern "C" int mocap_stage_timer_read(void* timer, float* ms_out)
{
    StageTimer* t = (StageTimer*)timer;
    if (!t || !ms_out) return MOCAP_ERR_INVALID;
    for (int i = 0; i < MOCAP_N_STAGES; ++i) {
        ms_out[i] = -1.0f;
        if (!t->recorded[i]) continue;
        CUDA_TRY(cudaEventSynchronize(t->ev[2 * i + 1]));
        CUDA_TRY(cudaEventElapsedTime(&ms_out[i], t->ev[2 * i], t->ev[2 * i + 1]));
    }
    return MOCAP_OK;
}

struct DetectLayout {
    size_t off_active, off_list, off_counters, off_bits, off_fg, off_nfg, off_flags, off_cellbox, off_blob, off_cluster;
    size_t blob_stride, total;
    ClusterLayout cl;
    int TX, TY, TXW, max_fg;
};

static int detect_layout(int n, int H, int W, int max_contours, int max_runs, bool with_blobs, DetectLayout* L)
{
    if (n <= 0 || H <= 0 || W <= 0) return MOCAP_ERR_INVALID;
    if (H > 16384 || W > 16384) return MOCAP_ERR_UNSUPPORTED;
    L->TX = cdiv(W, TILE); L->TY = cdiv(H, TILE); L->TXW = cdiv(L->TX, 32);
    L->max_fg = L->TX * L->TY;
    if ((long long)n * L->TX * L->TY >= (1LL << 31)) return MOCAP_ERR_UNSUPPORTED;   // tile codes are 32-bit
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t r = off; off += align_up(bytes, 256); return r; };
    L->off_active = take((size_t)n * L->TY * L->TXW * 4);
    L->off_list = take((size_t)n * L->TX * L->TY * 4);
    L->off_counters = take(64);
    L->off_bits = take((size_t)n * H * L->TX * 4);
    L->off_fg = take((size_t)n * L->max_fg * 4);
    L->off_nfg = take((size_t)n * 4);
    L->off_flags = take((size_t)n * 4);
    L->off_cellbox = take((size_t)n * L->TX * L->TY * 4);
    L->blob_stride = with_blobs ? blob_ws_stride(H, max_runs, max_contours) : 0;
    L->off_blob = take(L->blob_stride * (size_t)n);
    L->off_cluster = take(cluster_ws_bytes(n, H, W, max_contours, &L->cl));
    L->total = off;
    return MOCAP_OK;
}

static FilterWs filter_ws(char* base, const DetectLayout& L)
{
    FilterWs ws;
    ws.active = (uint32_t*)(base + L.off_active);
    ws.list = (uint32_t*)(base + L.off_list);
    ws.counters = (int*)(base + L.off_counters);
    ws.bits = (uint32_t*)(base + L.off_bits);
    ws.fg_tiles = (uint32_t*)(base + L.off_fg);
    ws.n_fg = (int*)(base + L.off_nfg);
    ws.cellbox = (uint32_t*)(base + L.off_cellbox);
    return ws;
}

extern "C" size_t mocap_detect_workspace_bytes(int n_frames, int H, int W, int max_blobs, int max_contours, int max_runs)
{
    (void)max_blobs;
    DetectLayout L;
    if (max_contours <= 0 || max_runs <= 0) return 0;
    if (detect_layout(n_frames, H, W, max_contours, max_runs, true, &L) != MOCAP_OK) return 0;
    return L.total;
}

extern "C" int mocap_filter_batch(const uint8_t* frames_dev, int n_frames, int H, int W, int64_t frame_stride,
                                  const void* table_dev, int thresh, uint32_t* out_bits,
                                  void* workspace, size_t workspace_bytes, void* stream)
{
    if (!frames_dev || !table_dev || !out_bits || !workspace) return MOCAP_ERR_INVALID;
    if (frame_stride < (int64_t)H * W) return MOCAP_ERR_INVALID;
    DetectLayout L;
    int st = detect_layout(n_frames, H, W, 1, 1, false, &L);
    if (st != MOCAP_OK) return st;
    if (workspace_bytes < L.total) return MOCAP_ERR_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    TableView tv; table_view(table_dev, H, W, &tv);
    FilterWs ws = filter_ws((char*)workspace, L);
    int* flags = (int*)((char*)workspace + L.off_flags);
    CUDA_TRY(cudaMemsetAsync(flags, 0, (size_t)n_frames * 4, s));
    st = launch_scan(frames_dev, n_frames, H, W, frame_stride, tv, thresh, ws, s, nullptr);
    if (st != MOCAP_OK) return st;
    st = launch_tiles(frames_dev, n_frames, H, W, frame_stride, tv, thresh, ws, L.max_fg, flags, nullptr, s);
    if (st != MOCAP_OK) return st;
    return launch_materialize_bits(ws, n_frames, H, W, tv, out_bits, s);
}

// The view of a lens set (MocapLensSet) for frames of H x W: the whole set is checked here, by every call that takes one
static int lens_set_view(const MocapLensSet* ls, int H, int W, TableView* tv)
{
    if (!ls || !ls->tables_dev || ls->n_lenses < 1) return MOCAP_ERR_INVALID;
    if (ls->lens_stride < mocap_undistort_table_bytes(H, W) || ls->lens_stride % 256 != 0) return MOCAP_ERR_INVALID;
    table_view(ls->tables_dev, H, W, tv);
    tv->lens_words = ls->lens_stride / 4;
    tv->n_lenses = ls->n_lenses;
    tv->frame_lens = ls->frame_lens_dev;
    return MOCAP_OK;
}

// mocap_detect_batch and mocap_detect_batch_subpixel: out_xy holds int32 (xy_float 0) or float32 (1) centroid pairs
static int detect_batch(const uint8_t* frames_dev, int n_frames, int H, int W, int64_t frame_stride,
                        const MocapLensSet* lenses, int thresh, double min_area, double min_circ,
                        int max_blobs, int max_contours, int max_runs,
                        int32_t* out_xy, int xy_float, int32_t* out_count, int32_t* out_flags,
                        uint32_t* out_bits, int32_t* out_labels, int64_t* out_blob_sums, int32_t* out_blob_count,
                        double* out_contours, int32_t* out_contour_count,
                        void* workspace, size_t workspace_bytes, void* stream, void* stage_timer)
{
    StageTimer* timer = (StageTimer*)stage_timer;
    if (!frames_dev || !out_xy || !out_count || !out_flags || !workspace) return MOCAP_ERR_INVALID;
    if (max_blobs <= 0 || max_contours <= 0 || max_runs <= 0) return MOCAP_ERR_INVALID;
    if (frame_stride < (int64_t)H * W) return MOCAP_ERR_INVALID;
    DetectLayout L;
    int st = detect_layout(n_frames, H, W, max_contours, max_runs, true, &L);
    if (st != MOCAP_OK) return st;
    TableView tv;
    st = lens_set_view(lenses, H, W, &tv);
    if (st != MOCAP_OK) return st;
    if (workspace_bytes < L.total) return MOCAP_ERR_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    FilterWs ws = filter_ws((char*)workspace, L);
    CUDA_TRY(cudaMemsetAsync(out_flags, 0, (size_t)n_frames * 4, s));
    if (out_labels) CUDA_TRY(cudaMemsetAsync(out_labels, 0, (size_t)n_frames * H * W * 4, s));
    // Product path (no label / bit-image outputs wanted): scan -> groups of hot cells -> per-cluster units in shared memory
    // -> per-frame ordering.  Frames it cannot finish locally, and every frame when the parity outputs are requested,
    // take the general per-frame path (tiles -> packed image -> runs, labels, contour tree).
    const bool extras = out_bits || out_labels || out_blob_sums || out_blob_count;
    const bool use_cluster = !extras && cluster_path_supported(H, W);
    char* cl_base = (char*)workspace + L.off_cluster;
    int* need_general = (int*)(cl_base + L.cl.need_general);
    st = launch_scan(frames_dev, n_frames, H, W, frame_stride, tv, thresh, ws, s, timer);
    if (st != MOCAP_OK) return st;
    CUDA_TRY(cudaMemsetAsync(need_general, use_cluster ? 0 : 1, (size_t)n_frames * 4, s));
    if (use_cluster) {
        st = launch_cluster_path(frames_dev, n_frames, H, W, frame_stride, tv, thresh, ws.cellbox, cl_base, L.cl, need_general,
                                 max_contours, max_blobs, min_area, min_circ, out_xy, xy_float, out_count, out_flags, out_contours,
                                 out_contour_count, s, timer, ClusterLaunch());
        if (st != MOCAP_OK) return st;
    }
    stage_begin(timer, 4, s);
    st = launch_tiles(frames_dev, n_frames, H, W, frame_stride, tv, thresh, ws, L.max_fg, out_flags, need_general, s);
    if (st != MOCAP_OK) return st;
    if (out_bits) {
        st = launch_materialize_bits(ws, n_frames, H, W, tv, out_bits, s);
        if (st != MOCAP_OK) return st;
    }
    st = launch_blobs(ws.bits, ws.fg_tiles, ws.n_fg, n_frames, H, W, L.TX, L.max_fg, max_runs, max_blobs, max_contours,
                      min_area, min_circ, (char*)workspace + L.off_blob, L.blob_stride,
                      out_xy, xy_float, out_count, out_flags, out_blob_sums, out_blob_count, out_contours, out_contour_count,
                      out_labels, need_general, s);
    stage_end(timer, 4, s);
    return st;
}

extern "C" int mocap_detect_batch(const uint8_t* frames_dev, int n_frames, int H, int W, int64_t frame_stride,
                                  const MocapLensSet* lenses, int thresh, double min_area, double min_circ,
                                  int max_blobs, int max_contours, int max_runs,
                                  int32_t* out_xy, int32_t* out_count, int32_t* out_flags,
                                  uint32_t* out_bits, int32_t* out_labels, int64_t* out_blob_sums, int32_t* out_blob_count,
                                  double* out_contours, int32_t* out_contour_count,
                                  void* workspace, size_t workspace_bytes, void* stream, void* stage_timer)
{
    return detect_batch(frames_dev, n_frames, H, W, frame_stride, lenses, thresh, min_area, min_circ, max_blobs, max_contours, max_runs,
                        out_xy, 0, out_count, out_flags, out_bits, out_labels, out_blob_sums, out_blob_count, out_contours, out_contour_count,
                        workspace, workspace_bytes, stream, stage_timer);
}

extern "C" int mocap_detect_batch_subpixel(const uint8_t* frames_dev, int n_frames, int H, int W, int64_t frame_stride,
                                           const MocapLensSet* lenses, int thresh, double min_area, double min_circ,
                                           int max_blobs, int max_contours, int max_runs,
                                           float* out_xy, int32_t* out_count, int32_t* out_flags,
                                           uint32_t* out_bits, int32_t* out_labels, int64_t* out_blob_sums, int32_t* out_blob_count,
                                           double* out_contours, int32_t* out_contour_count,
                                           void* workspace, size_t workspace_bytes, void* stream, void* stage_timer)
{
    return detect_batch(frames_dev, n_frames, H, W, frame_stride, lenses, thresh, min_area, min_circ, max_blobs, max_contours, max_runs,
                        (int32_t*)out_xy, 1, out_count, out_flags, out_bits, out_labels, out_blob_sums, out_blob_count, out_contours,
                        out_contour_count, workspace, workspace_bytes, stream, stage_timer);
}

// findContours -> filter -> moments on a given packed binary image (lib/ImageOperations.py:41-65), stage parity entry
extern "C" int mocap_blobs_batch(const uint32_t* bits_dev, int n_frames, int H, int W,
                                 double min_area, double min_circ, int max_blobs, int max_contours, int max_runs,
                                 int32_t* out_xy, int32_t* out_count, int32_t* out_flags,
                                 int32_t* out_labels, int64_t* out_blob_sums, int32_t* out_blob_count,
                                 double* out_contours, int32_t* out_contour_count,
                                 void* workspace, size_t workspace_bytes, void* stream)
{
    if (!bits_dev || !out_xy || !out_count || !out_flags || !workspace) return MOCAP_ERR_INVALID;
    if (max_blobs <= 0 || max_contours <= 0 || max_runs <= 0) return MOCAP_ERR_INVALID;
    DetectLayout L;
    int st = detect_layout(n_frames, H, W, max_contours, max_runs, true, &L);
    if (st != MOCAP_OK) return st;
    if (workspace_bytes < L.total) return MOCAP_ERR_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    FilterWs ws = filter_ws((char*)workspace, L);
    CUDA_TRY(cudaMemsetAsync(out_flags, 0, (size_t)n_frames * 4, s));
    if (out_labels) CUDA_TRY(cudaMemsetAsync(out_labels, 0, (size_t)n_frames * H * W * 4, s));
    st = launch_tiles_from_bits(bits_dev, n_frames, H, L.TX, L.TY, ws.fg_tiles, ws.n_fg, L.max_fg, s);
    if (st != MOCAP_OK) return st;
    return launch_blobs(bits_dev, ws.fg_tiles, ws.n_fg, n_frames, H, W, L.TX, L.max_fg, max_runs, max_blobs, max_contours,
                        min_area, min_circ, (char*)workspace + L.off_blob, L.blob_stride,
                        out_xy, 0, out_count, out_flags, out_blob_sums, out_blob_count, out_contours, out_contour_count,
                        out_labels, nullptr, s);
}


// =========================================================================================================
// Overlapped detection: the batch is cut into chunks of frames; the HBM-bound streaming scan of chunk k+1 runs
// beside the instruction-bound stages (group / piece filter / borders) of chunk k on the same SMs.  Chunk k's stages run as
// one chain on worker stream k mod workers.  The scan follows from the input:
//   cell boxes handed in (cellbox_dev): no scan.
//   frames a tensor map can describe, and stream memory operations available: ONE TMA-fed scan kernel over the whole batch
//     on the pipe's high-priority scan stream; it publishes a flag per finished chunk, which the chunk's worker stream waits
//     for with cuStreamWaitValue32 -- the scan CTA of an SM stays resident from the first byte to the last.
//   otherwise (and in the CPU emulation build, which has neither): the classic scan kernels chunk by chunk on the scan
//     stream, handed to the worker streams with one event per chunk.
// Whatever the cluster path hands to the general path is finished for the whole batch after the join.
// =========================================================================================================
#define PIPE_MAX_PROC 6
#define PIPE_MAX_CHUNKS 64
#define PIPE_TL_PER_CHUNK 4          // timeline marks per chunk: scan seen, grouped, filtered, borders done
#define PIPE_FILTER_CTAS_TMA 6       // persistent piece-filter CTAs per SM beside the TMA scan CTA
#define PIPE_FILTER_CTAS 8           // ... without it
#define PIPE_CAND_CTAS 12            // candidates_kernel CTAs per SM

// Store-to-peer epilogue of the multi-GPU pipeline: every frame's record (count + centroids) is copied to the address its consumer
// reads it from -- for the frame-sets of another rank that is a slot of THAT rank's receive buffer, mapped into this process
// (symmetric memory over NVLink), so the exchange step needs no collective, only a barrier.  One warp per frame.  phase 0 (after a
// chunk's border stage): frames the cluster path finished; phase 1 (after the general path): the frames it handed over.
__global__ void scatter_records_kernel(const int32_t* __restrict__ xy, const int32_t* __restrict__ count, const unsigned long long* __restrict__ xy_dst,
                                       const unsigned long long* __restrict__ count_dst, int n, int max_blobs, const int* __restrict__ need_general, int phase)
{
    const int lane = threadIdx.x & 31;
    const int f = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (f >= n) return;
    if ((need_general[f] != 0) != (phase != 0)) return;
    int c = count[f];
    c = c < 0 ? 0 : (c > max_blobs ? max_blobs : c);
    const uint2* src = (const uint2*)(xy + (size_t)f * max_blobs * 2);
    uint2* dst = (uint2*)xy_dst[f];
    for (int k = lane; k < c; k += 32) dst[k] = src[k];
    if (lane == 0) *(int32_t*)count_dst[f] = count[f];
}

static int launch_scatter(const int32_t* xy, const int32_t* count, const unsigned long long* xy_dst, const unsigned long long* count_dst,
                          int n, int max_blobs, const int* need_general, int phase, cudaStream_t s)
{
    LAUNCH(scatter_records_kernel, cdiv(n * 32, 128), 128, 0, s, xy, count, xy_dst, count_dst, n, max_blobs, need_general, phase);
    CUDA_TRY(cudaGetLastError());
    return MOCAP_OK;
}

// A pipe owns streams and events and remembers what its last call ran; everything a call reads is in its arguments.
struct DetectPipe {
    cudaStream_t s_scan = nullptr, s_proc[PIPE_MAX_PROC] = {};
    cudaEvent_t ev_fork = nullptr, ev_scan_done = nullptr, ev_proc_done[PIPE_MAX_PROC] = {}, ev_join = nullptr;
    cudaEvent_t ev_scan[PIPE_MAX_CHUNKS] = {};                       // classic scan: chunk c scanned
    cudaEvent_t ev_tl[PIPE_MAX_CHUNKS][PIPE_TL_PER_CHUNK] = {};      // timeline (timing enabled)
    int n_proc = 0;
    int tl_chunks = 0;               // chunks of the last call that recorded a timeline
    int last_tma = -1, last_chunks = 0;  // what the last call ran (mocap_detect_pipe_info)
};

extern "C" void* mocap_detect_pipe_create(int n_proc_streams)
{
    if (n_proc_streams < 1) n_proc_streams = 1;
    if (n_proc_streams > PIPE_MAX_PROC) n_proc_streams = PIPE_MAX_PROC;
    DetectPipe* p = new DetectPipe();
    p->n_proc = n_proc_streams;
    int lo = 0, hi = 0;
    bool ok = cudaDeviceGetStreamPriorityRange(&lo, &hi) == cudaSuccess;      // hi = numerically smallest = highest priority
    ok = ok && cudaStreamCreateWithPriority(&p->s_scan, cudaStreamNonBlocking, hi) == cudaSuccess;
    for (int i = 0; ok && i < n_proc_streams; ++i) ok = cudaStreamCreateWithPriority(&p->s_proc[i], cudaStreamNonBlocking, lo) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&p->ev_fork, cudaEventDefault) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&p->ev_scan_done, cudaEventDefault) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&p->ev_join, cudaEventDefault) == cudaSuccess;
    for (int i = 0; ok && i < n_proc_streams; ++i) ok = cudaEventCreateWithFlags(&p->ev_proc_done[i], cudaEventDisableTiming) == cudaSuccess;
    for (int c = 0; ok && c < PIPE_MAX_CHUNKS; ++c) {
        ok = cudaEventCreateWithFlags(&p->ev_scan[c], cudaEventDisableTiming) == cudaSuccess;
        for (int k = 0; ok && k < PIPE_TL_PER_CHUNK; ++k) ok = cudaEventCreateWithFlags(&p->ev_tl[c][k], cudaEventDefault) == cudaSuccess;
    }
    if (!ok) { delete p; return nullptr; }
    return p;
}

extern "C" void mocap_detect_pipe_destroy(void* pipe)
{
    DetectPipe* p = (DetectPipe*)pipe;
    if (!p) return;
    if (p->s_scan) cudaStreamDestroy(p->s_scan);
    for (int i = 0; i < PIPE_MAX_PROC; ++i) { if (p->s_proc[i]) cudaStreamDestroy(p->s_proc[i]); if (p->ev_proc_done[i]) cudaEventDestroy(p->ev_proc_done[i]); }
    if (p->ev_fork) cudaEventDestroy(p->ev_fork);
    if (p->ev_scan_done) cudaEventDestroy(p->ev_scan_done);
    if (p->ev_join) cudaEventDestroy(p->ev_join);
    for (int c = 0; c < PIPE_MAX_CHUNKS; ++c) {
        if (p->ev_scan[c]) cudaEventDestroy(p->ev_scan[c]);
        for (int k = 0; k < PIPE_TL_PER_CHUNK; ++k) if (p->ev_tl[c][k]) cudaEventDestroy(p->ev_tl[c][k]);
    }
    delete p;
}

struct PipeLayout {
    DetectLayout L;                  // general-path arrays of the whole batch (its cluster part serves chunk 0 .. see below)
    size_t off_ctrl, off_need, off_chunks, chunk_bytes, total;
    ClusterLayout cl;                // inside one chunk's cluster workspace
    int chunks, chunk_frames;
};

static int pipe_layout(int n, int H, int W, int max_contours, int max_runs, int chunk_frames, PipeLayout* P)
{
    if (chunk_frames <= 0 || chunk_frames > n) chunk_frames = n;
    int chunks = cdiv(n, chunk_frames);
    if (chunks > PIPE_MAX_CHUNKS) { chunk_frames = cdiv(n, PIPE_MAX_CHUNKS); chunks = cdiv(n, chunk_frames); }
    P->chunks = chunks; P->chunk_frames = chunk_frames;
    int st = detect_layout(n, H, W, max_contours, max_runs, true, &P->L);
    if (st != MOCAP_OK) return st;
    size_t off = P->L.off_cluster;                                  // the whole-batch cluster workspace is replaced by the per-chunk ones
    auto take = [&](size_t bytes) { size_t r = off; off += align_up(bytes, 256); return r; };
    P->off_ctrl = take(scan_tma_ctrl_bytes(chunks));
    P->off_need = take((size_t)n * 4);
    P->chunk_bytes = align_up(cluster_ws_bytes(chunk_frames, H, W, max_contours, &P->cl), 256);
    P->off_chunks = take(P->chunk_bytes * (size_t)chunks);
    P->total = off > P->L.total ? off : P->L.total;
    return MOCAP_OK;
}

extern "C" size_t mocap_detect_pipelined_workspace_bytes(int n_frames, int H, int W, int max_blobs, int max_contours, int max_runs, int chunk_frames)
{
    (void)max_blobs;
    if (max_contours <= 0 || max_runs <= 0) return 0;
    PipeLayout P;
    if (pipe_layout(n_frames, H, W, max_contours, max_runs, chunk_frames, &P) != MOCAP_OK) return 0;
    return P.total;
}

// mocap_detect_batch_pipelined and mocap_detect_batch_pipelined_subpixel: int32 (xy_float 0) or float32 (1) centroid pairs.  The
// store-to-peer epilogue copies 8-byte records and does not care which.
static int detect_pipelined(void* pipe, const uint8_t* frames_dev, int n_frames, int H, int W, int64_t frame_stride,
                            const MocapLensSet* lenses, int thresh, double min_area, double min_circ,
                            int max_blobs, int max_contours, int max_runs,
                            int32_t* out_xy, int xy_float, int32_t* out_count, int32_t* out_flags,
                            double* out_contours, int32_t* out_contour_count,
                            const uint32_t* cellbox_dev, const uint64_t* xy_dst_dev, const uint64_t* count_dst_dev,
                            void* scan_wait_event, void* scan_done_event,
                            void* workspace, size_t workspace_bytes, void* stream, int chunk_frames, int record_timeline)
{
    DetectPipe* dp = (DetectPipe*)pipe;
    if (!dp || !frames_dev || !out_xy || !out_count || !out_flags || !workspace) return MOCAP_ERR_INVALID;
    if ((xy_dst_dev == nullptr) != (count_dst_dev == nullptr)) return MOCAP_ERR_INVALID;
    if (max_blobs <= 0 || max_contours <= 0 || max_runs <= 0) return MOCAP_ERR_INVALID;
    if (frame_stride < (int64_t)H * W) return MOCAP_ERR_INVALID;
    PipeLayout P;
    int st = pipe_layout(n_frames, H, W, max_contours, max_runs, chunk_frames, &P);
    if (st != MOCAP_OK) return st;
    TableView tv;
    st = lens_set_view(lenses, H, W, &tv);
    if (st != MOCAP_OK) return st;
    if (workspace_bytes < P.total) return MOCAP_ERR_WORKSPACE;
    if (!cluster_path_supported(H, W)) return MOCAP_ERR_UNSUPPORTED;         // such shapes take mocap_detect_batch
    cudaStream_t s = (cudaStream_t)stream;
    const unsigned long long* sc_xy = (const unsigned long long*)xy_dst_dev;
    const unsigned long long* sc_count = (const unsigned long long*)count_dst_dev;
    char* base = (char*)workspace;
    FilterWs ws = filter_ws(base, P.L);
    // hot cell boxes handed in (the Bayer front step computes them while it writes the grey frames): no streaming scan in this call
    const bool prescanned = cellbox_dev != nullptr;
    if (prescanned) ws.cellbox = (uint32_t*)cellbox_dev;
    int* ctrl = (int*)(base + P.off_ctrl);
    int* need_general = (int*)(base + P.off_need);
    const int chunks = P.chunks, cf = P.chunk_frames;
    const bool tma = !prescanned && scan_tma_supported(frames_dev, n_frames, H, W, frame_stride, thresh) && stream_wait_supported();
    dp->last_tma = tma ? 1 : 0; dp->last_chunks = chunks;
    dp->tl_chunks = 0;
    ClusterLaunch how;
    how.zero = 0;                    // the chunk loop clears each chunk's block on its worker stream ahead of its scan wait
    how.filter_ctas = tma ? PIPE_FILTER_CTAS_TMA : PIPE_FILTER_CTAS;
    how.cand_ctas = PIPE_CAND_CTAS;
    CUDA_TRY(cudaMemsetAsync(out_flags, 0, (size_t)n_frames * 4, s));
    CUDA_TRY(cudaMemsetAsync(need_general, 0, (size_t)n_frames * 4, s));
    CUDA_TRY(cudaMemsetAsync(ctrl, 0, scan_tma_ctrl_bytes(chunks), s));
    CUDA_TRY(cudaEventRecord(dp->ev_fork, s));
    CUDA_TRY(cudaStreamWaitEvent(dp->s_scan, dp->ev_fork, 0));
    if (scan_wait_event) CUDA_TRY(cudaStreamWaitEvent(dp->s_scan, (cudaEvent_t)scan_wait_event, 0));    // scans of several pipes one after the other
    if (tma) {
        st = launch_scan_tma(frames_dev, n_frames, H, W, frame_stride, tv, thresh, ws.cellbox, ctrl, chunks, cf, dp->s_scan);
        if (st != MOCAP_OK) return st;
    }
    for (int i = 0; i < dp->n_proc; ++i) CUDA_TRY(cudaStreamWaitEvent(dp->s_proc[i], dp->ev_fork, 0));
    for (int c = 0; c < chunks; ++c) {
        const int f0 = c * cf, nc = (n_frames - f0) < cf ? (n_frames - f0) : cf;
        cudaStream_t ps = dp->s_proc[c % dp->n_proc];
        char* cws = base + P.off_chunks + (size_t)c * P.chunk_bytes;
        uint32_t* cb = ws.cellbox + (size_t)f0 * tv.TX * tv.TY;
        CUDA_TRY(cudaMemsetAsync(cws + P.cl.zero_begin, 0, P.cl.zero_bytes, ps));     // the chunk's counters / lists, off the critical path
        if (tma) {
            st = stream_wait_geq(ps, scan_tma_chunk_flag(ctrl, chunks, c), 1);
            if (st != MOCAP_OK) return st;
        } else if (!prescanned) {                                                   // (handed-in boxes were complete before the fork)
            FilterWs wc = ws; wc.cellbox = cb;
            st = launch_scan(frames_dev + (size_t)f0 * frame_stride, nc, H, W, frame_stride, tv, thresh, wc, dp->s_scan, nullptr);
            if (st != MOCAP_OK) return st;
            CUDA_TRY(cudaEventRecord(dp->ev_scan[c], dp->s_scan));
            CUDA_TRY(cudaStreamWaitEvent(ps, dp->ev_scan[c], 0));
        }
        if (record_timeline) CUDA_TRY(cudaEventRecord(dp->ev_tl[c][0], ps));
        how.ev_group = dp->ev_tl[c][1]; how.ev_filter = dp->ev_tl[c][2]; how.ev_borders = dp->ev_tl[c][3];
        TableView tc = tv;                                                          // the chunk's frames are numbered from 0
        if (tc.frame_lens) tc.frame_lens += f0;
        st = launch_cluster_path(frames_dev + (size_t)f0 * frame_stride, nc, H, W, frame_stride, tc, thresh, cb, cws, P.cl, need_general + f0,
                                 max_contours, max_blobs, min_area, min_circ,
                                 out_xy + (size_t)f0 * max_blobs * 2, xy_float, out_count + f0, out_flags + f0,
                                 out_contours ? out_contours + (size_t)f0 * max_contours * 8 : nullptr, out_contour_count ? out_contour_count + f0 : nullptr,
                                 ps, nullptr, how);
        if (st != MOCAP_OK) return st;
        if (sc_xy) {                                         // the chunk's records go where their consumers read them, off the critical path
            st = launch_scatter(out_xy + (size_t)f0 * max_blobs * 2, out_count + f0, sc_xy + f0, sc_count + f0, nc, max_blobs, need_general + f0, 0, ps);
            if (st != MOCAP_OK) return st;
        }
    }
    CUDA_TRY(cudaEventRecord(dp->ev_scan_done, dp->s_scan));
    if (scan_done_event) CUDA_TRY(cudaEventRecord((cudaEvent_t)scan_done_event, dp->s_scan));
    CUDA_TRY(cudaStreamWaitEvent(s, dp->ev_scan_done, 0));
    for (int i = 0; i < dp->n_proc; ++i) {
        CUDA_TRY(cudaEventRecord(dp->ev_proc_done[i], dp->s_proc[i]));
        CUDA_TRY(cudaStreamWaitEvent(s, dp->ev_proc_done[i], 0));
    }
    if (record_timeline) { CUDA_TRY(cudaEventRecord(dp->ev_join, s)); dp->tl_chunks = chunks; }
    // general path for the frames the cluster units could not finish (rare), whole batch
    st = launch_tiles(frames_dev, n_frames, H, W, frame_stride, tv, thresh, ws, P.L.max_fg, out_flags, need_general, s);
    if (st != MOCAP_OK) return st;
    st = launch_blobs(ws.bits, ws.fg_tiles, ws.n_fg, n_frames, H, W, P.L.TX, P.L.max_fg, max_runs, max_blobs, max_contours,
                      min_area, min_circ, base + P.L.off_blob, P.L.blob_stride,
                      out_xy, xy_float, out_count, out_flags, nullptr, nullptr, out_contours, out_contour_count, nullptr, need_general, s);
    if (st == MOCAP_OK && sc_xy) st = launch_scatter(out_xy, out_count, sc_xy, sc_count, n_frames, max_blobs, need_general, 1, s);
    return st;
}

extern "C" int mocap_detect_batch_pipelined(void* pipe, const uint8_t* frames_dev, int n_frames, int H, int W, int64_t frame_stride,
                                            const MocapLensSet* lenses, int thresh, double min_area, double min_circ,
                                            int max_blobs, int max_contours, int max_runs,
                                            int32_t* out_xy, int32_t* out_count, int32_t* out_flags,
                                            double* out_contours, int32_t* out_contour_count,
                                            const uint32_t* cellbox_dev, const uint64_t* xy_dst_dev, const uint64_t* count_dst_dev,
                                            void* scan_wait_event, void* scan_done_event,
                                            void* workspace, size_t workspace_bytes, void* stream, int chunk_frames, int record_timeline)
{
    return detect_pipelined(pipe, frames_dev, n_frames, H, W, frame_stride, lenses, thresh, min_area, min_circ, max_blobs, max_contours,
                            max_runs, out_xy, 0, out_count, out_flags, out_contours, out_contour_count, cellbox_dev, xy_dst_dev,
                            count_dst_dev, scan_wait_event, scan_done_event, workspace, workspace_bytes, stream, chunk_frames, record_timeline);
}

extern "C" int mocap_detect_batch_pipelined_subpixel(void* pipe, const uint8_t* frames_dev, int n_frames, int H, int W, int64_t frame_stride,
                                                     const MocapLensSet* lenses, int thresh, double min_area, double min_circ,
                                                     int max_blobs, int max_contours, int max_runs,
                                                     float* out_xy, int32_t* out_count, int32_t* out_flags,
                                                     double* out_contours, int32_t* out_contour_count,
                                                     const uint32_t* cellbox_dev, const uint64_t* xy_dst_dev, const uint64_t* count_dst_dev,
                                                     void* scan_wait_event, void* scan_done_event,
                                                     void* workspace, size_t workspace_bytes, void* stream, int chunk_frames, int record_timeline)
{
    return detect_pipelined(pipe, frames_dev, n_frames, H, W, frame_stride, lenses, thresh, min_area, min_circ, max_blobs, max_contours,
                            max_runs, (int32_t*)out_xy, 1, out_count, out_flags, out_contours, out_contour_count, cellbox_dev, xy_dst_dev,
                            count_dst_dev, scan_wait_event, scan_done_event, workspace, workspace_bytes, stream, chunk_frames, record_timeline);
}

// Timeline of the last mocap_detect_batch_pipelined call that had record_timeline set (read it after the stream has been
// synchronised): ms since the fork for [scan kernel(s) done, join] followed by, per chunk, [scan seen, grouped, filtered,
// borders done].  Returns the number of floats written (2 + 4 chunks), 0 if there is no timeline, or a negative status.
extern "C" int mocap_detect_pipe_timeline(void* pipe, float* ms_out, int cap)
{
    DetectPipe* dp = (DetectPipe*)pipe;
    if (!dp || !ms_out) return MOCAP_ERR_INVALID;
    const int need = 2 + PIPE_TL_PER_CHUNK * dp->tl_chunks;
    if (dp->tl_chunks == 0) return 0;
    if (cap < need) return MOCAP_ERR_INVALID;
    CUDA_TRY(cudaEventSynchronize(dp->ev_join));
    CUDA_TRY(cudaEventElapsedTime(&ms_out[0], dp->ev_fork, dp->ev_scan_done));
    CUDA_TRY(cudaEventElapsedTime(&ms_out[1], dp->ev_fork, dp->ev_join));
    for (int c = 0; c < dp->tl_chunks; ++c)
        for (int k = 0; k < PIPE_TL_PER_CHUNK; ++k)
            CUDA_TRY(cudaEventElapsedTime(&ms_out[2 + c * PIPE_TL_PER_CHUNK + k], dp->ev_fork, dp->ev_tl[c][k]));
    return need;
}

// what the last pipelined call actually ran: [0] scan kernel (1 = TMA ring, the workers waited on its chunk flags; 0 = classic or
// none), [1] chunks
extern "C" int mocap_detect_pipe_info(void* pipe, int* out2)
{
    DetectPipe* dp = (DetectPipe*)pipe;
    if (!dp || !out2) return MOCAP_ERR_INVALID;
    out2[0] = dp->last_tma; out2[1] = dp->last_chunks;
    return MOCAP_OK;
}

// the streaming scan alone (stage parity): cellbox_out [n][TY][TX] packed hot boxes (x0 | x1 << 8 | y0 << 16 | y1 << 24,
// 0xffffffff = no pixel > thresh in the cell).  variant 0: classic register-staged kernels, 1: TMA ring.
extern "C" int mocap_scan_cells_batch(const uint8_t* frames_dev, int n_frames, int H, int W, int64_t frame_stride, const void* table_dev,
                                      int thresh, int variant, uint32_t* cellbox_out, void* workspace, size_t workspace_bytes, void* stream)
{
    if (!frames_dev || !table_dev || !cellbox_out || n_frames <= 0 || H <= 0 || W <= 0) return MOCAP_ERR_INVALID;
    if (frame_stride < (int64_t)H * W || (variant != 0 && variant != 1)) return MOCAP_ERR_INVALID;
    cudaStream_t s = (cudaStream_t)stream;
    TableView tv; table_view(table_dev, H, W, &tv);
    if (variant == 0) {
        FilterWs ws; memset(&ws, 0, sizeof(ws));
        ws.cellbox = cellbox_out;
        return launch_scan(frames_dev, n_frames, H, W, frame_stride, tv, thresh, ws, s, nullptr);
    }
    if (!scan_tma_supported(frames_dev, n_frames, H, W, frame_stride, thresh)) return MOCAP_ERR_UNSUPPORTED;
    if (!workspace || workspace_bytes < scan_tma_ctrl_bytes(1)) return MOCAP_ERR_WORKSPACE;
    CUDA_TRY(cudaMemsetAsync(workspace, 0, scan_tma_ctrl_bytes(1), s));
    return launch_scan_tma(frames_dev, n_frames, H, W, frame_stride, tv, thresh, cellbox_out, (int*)workspace, 1, n_frames, s);
}
