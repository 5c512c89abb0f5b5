// Shared device/host helpers for libmocap_b200 (sm_100a only).
#pragma once
#ifdef MOCAP_EMU
// tests/emu builds this same source with g++ for the GPU-less CPU test-suite (never part of the product library)
#include "cuda_emu.h"
#define LAUNCH(kernel, grid, block, smem, stream, ...) \
    (mocap_count_launch(), emu::launch(dim3(grid), dim3(block), (size_t)(smem), [=]() { kernel(__VA_ARGS__); }))
#define DYN_SHARED(name) unsigned char* name = emu::dyn_smem()
// the overlapped detection's streams and events there: launches run where they are issued, so every stream is the null
// stream and waiting for an event has nothing to wait for
enum { cudaStreamNonBlocking = 1, cudaEventDefault = 0, cudaEventDisableTiming = 2 };
static inline cudaError_t cudaEventCreateWithFlags(cudaEvent_t* e, unsigned) { return cudaEventCreate(e); }
static inline cudaError_t cudaDeviceGetStreamPriorityRange(int* lo, int* hi) { *lo = 0; *hi = 0; return 0; }
static inline cudaError_t cudaStreamCreateWithPriority(cudaStream_t* s, unsigned, int) { *s = nullptr; return 0; }
static inline cudaError_t cudaStreamDestroy(cudaStream_t) { return 0; }
static inline cudaError_t cudaStreamWaitEvent(cudaStream_t, cudaEvent_t, unsigned) { return 0; }
#else
#include <cuda_runtime.h>
#define LAUNCH(kernel, grid, block, smem, stream, ...) (mocap_count_launch(), kernel<<<grid, block, smem, stream>>>(__VA_ARGS__))
#define DYN_SHARED(name) extern __shared__ __align__(16) unsigned char name[]
#endif
#include <stdint.h>
#include "../../include/mocap_b200.h"

#define MOCAP_ABI_VERSION 6

// every kernel launch of the library is counted (mocap_kernel_launch_count: the bench's gpu_launches is read, not estimated)
extern unsigned long long g_mocap_launches;
static inline void mocap_count_launch() { __atomic_fetch_add(&g_mocap_launches, 1ull, __ATOMIC_RELAXED); }

#define TILE 32              // output tile edge (pixels) == bits per packed word
#define HALO_U 4             // undistorted pixels needed around an output tile (2 blur + 2 majority)
#define REG_U (TILE + 2 * HALO_U)   // 40
#define REG_B (TILE + 4)            // 36

#define CUDA_TRY(expr)                                  \
    do {                                                \
        cudaError_t _e = (expr);                        \
        if (_e != cudaSuccess) return MOCAP_ERR_CUDA;   \
    } while (0)

static inline int cdiv(int a, int b) { return (a + b - 1) / b; }
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ---------------------------------------------------------------------------------------------------------
// Undistortion table (built by mocap_undistort_table_build, consumed by the detection kernels)
// ---------------------------------------------------------------------------------------------------------
struct TableHeader {
    uint32_t magic;
    int32_t H, W;
    int32_t TX, TY;          // output tiles (32x32) == source cells
    int32_t overflow;        // a displacement did not fit the int16 fixed-point encoding
    int32_t n_zero;          // pixels whose source lies fully outside the frame
    int32_t pad;
    uint64_t off_map;        // int32 [H][W]: low16 = iu - 32*x, high16 = iv - 32*y (1/32 px), 0x80008000 = outside
    uint64_t off_cell;       // int32 [TY][TX][4]: output-tile rectangle (tx0,ty0,tx1,ty1) that samples this source cell
    uint64_t off_tile;       // int32 [TY][TX][8]: source box sx0,sy0,sx1,sy1 and displacement bounds dxmin,dxmax,dymin,dymax
    uint64_t off_cellinv;    // int32 [TY][TX][4]: bounds dxmin,dxmax,dymin,dymax of (source - output) over every output pixel that can sample the cell
    uint64_t off_fast;       // int32 [H][W] (+ 16 bytes): the map in the form the piece filter consumes: fx | fy << 8 | tap offset << 16, where
                             // tap offset = (dv >> 5) * WIN_W + (du >> 5) is where the pixel's first tap lies in a staged source window relative to the
                             // pixel's own place in it; FAST_INVALID where the pixel maps outside or the offset does not fit 16 bits
    uint64_t off_tflag;      // int32 [TY][TX]: != 0 when an output pixel of the tile has no valid fast-map entry
    uint64_t total_bytes;
};
#define TABLE_MAGIC 0x4d43424bu
#define MAP_OUTSIDE 0x80008000u
#define WIN_W 96             // row stride of the staged source window of a filter piece (detect_cluster.cu); the fast map is built for it
#define FAST_INVALID 0x80000000u

// The arrays of lens 0; lens l's table lies l * lens_words int32 words further (a lens set, MocapLensSet).
struct TableView {
    const int32_t* map;
    const int32_t* cell;
    const int32_t* tile;
    const int32_t* cellinv;
    const int32_t* fast;
    const int32_t* tflag;
    int H, W, TX, TY;
    size_t lens_words;           // lens_stride / 4 (0 with one table)
    int n_lenses;
    const int32_t* frame_lens;   // [n] lens of every frame of the call, or null: lens 0
};

// Lens of frame f, -1 when its index lies outside [0, n_lenses) (the frame is flagged MOCAP_FLAG_LENS_INDEX and no table is read
// for it).  Read once per frame, by the kernel that first reads the frame's table.
__device__ __forceinline__ int frame_lens_of(const TableView& tv, int f)
{
    if (!tv.frame_lens) return 0;
    const int l = tv.frame_lens[f];
    return (unsigned)l < (unsigned)tv.n_lenses ? l : -1;
}
// tv with its arrays moved to lens l's table
__device__ __forceinline__ TableView lens_table(TableView tv, int l)
{
    const size_t o = (size_t)l * tv.lens_words;
    tv.map += o; tv.cell += o; tv.tile += o; tv.cellinv += o; tv.fast += o; tv.tflag += o;
    return tv;
}

// per-stage CUDA events of one mocap_detect_batch call (mocap_stage_timer_*)
struct StageTimer {
    cudaEvent_t ev[2 * MOCAP_N_STAGES];
    int recorded[MOCAP_N_STAGES];
};
static inline void stage_begin(StageTimer* t, int stage, cudaStream_t s) { if (t) { cudaEventRecord(t->ev[2 * stage], s); } }
static inline void stage_end(StageTimer* t, int stage, cudaStream_t s) { if (t) { cudaEventRecord(t->ev[2 * stage + 1], s); t->recorded[stage] = 1; } }

#define CELL_EMPTY 0xffffffffu
// ---------------------------------------------------------------------------------------------------------
// hot-pixel test: byte > thresh, four bytes at a time.  T = thresh + 1.
//   T in 129..255: bit7(b) & bit7((b & 0x7f) + (256 - T));   T in 1..128: bit7(b) | bit7((b & 0x7f) + (128 - T))
// ---------------------------------------------------------------------------------------------------------
struct HotTest { uint32_t add; int mode; };   // mode 0: and, 1: or, 2: never, 3: always
static inline HotTest make_hot_test(int thresh)
{
    HotTest h; int T = thresh + 1;
    if (T >= 256) { h.mode = 2; h.add = 0; }
    else if (T <= 0) { h.mode = 3; h.add = 0; }
    else if (T > 128) { h.mode = 0; h.add = 0x01010101u * (uint32_t)(256 - T); }
    else { h.mode = 1; h.add = 0x01010101u * (uint32_t)(128 - T); }
    return h;
}
template <int MODE>
__device__ __forceinline__ uint32_t hot4(uint32_t w, uint32_t add)
{
    uint32_t t = (w & 0x7f7f7f7fu) + add;
    if (MODE == 0) return w & t;        // caller masks with 0x80808080
    if (MODE == 1) return w | t;
    if (MODE == 2) return 0u;
    return 0x80808080u;
}

// hot byte lanes of a 32-bit word (bit 7 of every byte of h) -> 4-bit mask, bit b = byte b
__device__ __forceinline__ uint32_t hot_nibble(uint32_t h)
{
    h &= 0x80808080u;
    return ((h >> 7) | (h >> 14) | (h >> 21) | (h >> 28)) & 0xfu;
}

// cell-local hot bounding box packed x0 | x1 << 8 | y0 << 16 | y1 << 24; CELL_EMPTY when the cell holds no pixel > thresh
__device__ __forceinline__ uint32_t pack_cellbox(uint32_t xmask, uint32_t ymask)
{
    if (!xmask) return CELL_EMPTY;
    uint32_t x0 = __ffs(xmask) - 1, x1 = 31 - __clz(xmask), y0 = __ffs(ymask) - 1, y1 = 31 - __clz(ymask);
    return x0 | (x1 << 8) | (y0 << 16) | (y1 << 24);
}

// The centroid record of a kept contour: (m10 / m00, m01 / m00) as the FP64 quotients of cv.moments, stored in the 8-byte slot
// xy[0..1] as int32 truncated toward zero (int(), lib/ImageOperations.py:59-62) or, sub-pixel, as the float32 nearest to them.
__device__ __forceinline__ void store_centroid(int32_t* xy, double qx, double qy, int xy_float)
{
    if (xy_float) { float* p = (float*)xy; p[0] = (float)qx; p[1] = (float)qy; }
    else { xy[0] = (int32_t)qx; xy[1] = (int32_t)qy; }
}

// The reference's filter of a border (lib/ImageOperations.py:43-51) from its Green sum a00 (twice the signed area) and its
// perimeter: circularity 4 pi area / perimeter^2 > min_circ and area > min_area, and m00 != 0 (a centroid exists).
__device__ __forceinline__ int contour_keep(long long a00, double per, double min_area, double min_circ)
{
    const double area = (double)(a00 < 0 ? -a00 : a00) * 0.5;
    int keep = 0;
    if (per != 0.0) {
        const double circ = __ddiv_rn(__dmul_rn(12.566370614359172, area), __dmul_rn(per, per));
        keep = (circ > min_circ && area > min_area) ? 1 : 0;
    }
    return a00 == 0 ? 0 : keep;
}

// The centroid record of a kept border from its Green sums: cv.moments' m00, m10, m01 (a00 / 2, a10 / 6, a01 / 6 with the sign
// of a00), then store_centroid.
__device__ __forceinline__ void store_blob_centroid(int32_t* xy, long long a00, long long a10, long long a01, int xy_float)
{
    const double sgn = a00 > 0 ? 1.0 : -1.0;
    const double m00 = __dmul_rn((double)a00, sgn * 0.5);
    const double m10 = __dmul_rn((double)a10, sgn * 0.16666666666666666);
    const double m01 = __dmul_rn((double)a01, sgn * 0.16666666666666666);
    store_centroid(xy, __ddiv_rn(m10, m00), __ddiv_rn(m01, m00), xy_float);
}

// how launch_cluster_path runs one chunk of frames
struct ClusterLaunch {
    int filter_ctas;                 // persistent piece-filter CTAs per SM (fewer when the TMA scan is co-resident)
    int cand_ctas;                   // candidates_kernel CTAs per SM
    cudaEvent_t ev_group = nullptr, ev_filter = nullptr, ev_borders = nullptr;   // recorded after the stages (timeline marks)
};

// byte offsets of the cluster path's arrays in its workspace (cluster_ws_bytes)
struct ClusterLayout {
    size_t zero_bytes;               // the first bytes, which the caller zeroes before the launch: counters, rec_count, cand_count, frame_clusters
    size_t counters, rec_count, cand_count, frame_clusters;
    size_t clusters, pieces, rec_start, rec_a, rec_per, memb, rows_out, cand_list, rec_info;
};

// workspace slices of the filter stage (carved by api.cu)
struct FilterWs {
    uint32_t* active;    // [n][TY][TXW] bitmap of output tiles that can hold foreground
    uint32_t* list;      // [n * TX * TY] work list: frame * (TX*TY) + tile
    int* counters;       // [0] = list length, [1] = work cursor
    uint32_t* bits;      // [n][H][TX] packed binary image (only active tiles and their neighbours are defined)
    uint32_t* fg_tiles;  // [n][max_fg] tiles that hold at least one foreground pixel
    int* n_fg;           // [n]
    uint32_t* cellbox;   // [n][TY][TX] hot bounding box of every 32x32 source cell (written by the scan pass)
};

// 8-neighbour codes: 0=E 1=NE 2=N 3=NW 4=W 5=SW 6=S 7=SE (y grows downwards)
// dx+1 = {2,2,1,0,0,0,1,2}, dy+1 = {1,0,0,0,1,2,2,2} packed two bits per direction
__device__ __forceinline__ int dir_dx(int d) { return ((0x901A >> (2 * d)) & 3) - 1; }
__device__ __forceinline__ int dir_dy(int d) { return ((0xA901 >> (2 * d)) & 3) - 1; }
