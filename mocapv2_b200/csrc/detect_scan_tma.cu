// Streaming scan of _find_dot's detection, TMA-fed (sm_100a): the pass that reads every frame byte once and leaves the hot
// bounding box of every 32x32 source cell (cellbox), see detect_filter.cu for what "hot" means and why that is all the later
// stages need (lib/ImageOperations.py:38-40 of the reference: undistort -> blur -> threshold -> median can only set a pixel
// within reach of a source byte > thresh).
//
// Why a second scan kernel: scan_hot_vec32_kernel keeps its bytes in flight in REGISTERS (256 threads x 64 registers x 4 CTAs
// = the whole register file of an SM), so nothing else can run beside it, although it needs less than half of the issue
// slots.  Here the bytes in flight live in SHARED MEMORY: one producer thread per SM posts 256x32-byte boxes of the frame
// batch, viewed as a 3-D tensor [n][H][W] of u8, into a ring of ST_STAGES x 8 KB with cp.async.bulk.tensor.3d (TMA, L2
// evict-first: the frames are read once) completing on mbarriers; ST_CONSUMERS warps test the boxes out of shared memory with
// 128-bit loads (conflict-free: a quarter warp reads 128 consecutive bytes).  One CTA of 160 threads x <= 48 registers + 49 KB
// per SM leaves six of the eight piece-filter CTAs, and every other kernel of the path, room on the same SM: the HBM-bound
// scan of chunk k+1 runs under the instruction-bound stages of chunk k (api.cu, mocap_detect_batch_pipelined).
// Rows / columns beyond the frame are zero-filled by the TMA unit, so ragged frame sizes need no edge code; what the tensor
// map cannot describe (rows that are not a multiple of 16 bytes, thresholds outside 0..254) stays with the classic kernels.
//
// Progress is published per CHUNK of frames: a consumer warp counts the boxes it finished per chunk and adds them to
// chunk_done[]; the warp that completes a chunk sets chunk_flag[chunk], which the host side waits for with a stream
// memory operation (cuStreamWaitValue32) -- no kernel ever spins on another kernel.
#include "common.cuh"

// Control block of a launch: int [SCAN_CTRL_WORK + 2 chunks] = the work counter (slot 0, the rest of the head is unused), then
// chunk_done[], chunk_flag[].
#define SCAN_CTRL_WORK 64
size_t scan_tma_ctrl_bytes(int chunks) { return align_up((size_t)(SCAN_CTRL_WORK + 2 * chunks) * 4, 256); }
const int* scan_tma_chunk_flag(const int* ctrl, int chunks, int chunk) { return ctrl + SCAN_CTRL_WORK + chunks + chunk; }

#include "tma.cuh"
#ifndef MOCAP_EMU

#define ST_BOX_W 256
#define ST_BOX_H 32
#define ST_STAGE_BYTES (ST_BOX_W * ST_BOX_H)
#define ST_CONSUMERS 4
#define ST_STAGES 6                // ring slots of 8 KB
#define ST_GRAB 8                  // boxes a producer draws from the work counter at a time (one 2048-pixel band of cells)
#define ST_THREADS (32 * (ST_CONSUMERS + 1))

struct ScanTmaArgs {
    uint32_t* cellbox;             // [n][TY][TX]
    int* work;                     // work counter of this launch (boxes handed out, relative to item_begin)
    int* chunk_done;               // [chunks] boxes finished
    int* chunk_flag;               // [chunks] 1 when all boxes of the chunk are finished
    int TX, TY, XB;                // cells per row / column, boxes per cell row
    int items_per_chunk, item_begin, item_end, total_items;
    uint32_t add;                  // SWAR constant of the hot test (make_hot_test)
};
struct __align__(16) StageRec { int cb_index, ncell, chunk, pad; };

// publish `cnt` finished boxes of chunk `ch` (whole warp calls; every cellbox store of those boxes precedes it)
__device__ __forceinline__ void scan_publish(const ScanTmaArgs& a, int ch, int cnt, int lane)
{
    if (cnt <= 0) return;
    __syncwarp();
    if (lane == 0) {
        __threadfence();
        const int in_chunk = min(a.items_per_chunk, a.total_items - ch * a.items_per_chunk);
        const int old = atomicAdd(&a.chunk_done[ch], cnt);
        if (old + cnt == in_chunk) { __threadfence_system(); atomicExch(&a.chunk_flag[ch], 1); }
    }
}

template <int MODE>
__global__ void __launch_bounds__(ST_THREADS, 8) scan_tma_kernel(const __grid_constant__ CUtensorMap tmap, ScanTmaArgs a)
{
    extern __shared__ unsigned char st_raw[];
    unsigned char* st = st_raw + ((128u - (smem_u32(st_raw) & 127u)) & 127u);          // TMA destinations: 128-byte aligned
    uint8_t* ring = st;
    // "box landed" barriers: NB per ring slot, used by successive fills in turn.  Consumer warps take the boxes round-robin, so
    // successive fills of a slot are waited for by different warps, and TMA completions arrive out of order: a warp that has finished
    // box q starts waiting for box q + C (C consumer warps) while older boxes may still be in flight -- if the barrier it waits on were
    // still in the phase of an older, unfinished fill, its parity test would pass at once (parity only tells odd from even phases).
    // A barrier is reused every NB * S boxes (S slots); its previous fill q + C - NB * S is certainly complete when box q has been
    // ISSUED (its slot was handed back before box q + C - (NB - 1) * S went into it), i.e. when C <= (NB - 1) * S.
    constexpr int NB = (ST_CONSUMERS + ST_STAGES - 1) / ST_STAGES + 1;
    uint64_t* full = (uint64_t*)(st + ST_STAGES * ST_STAGE_BYTES);
    uint64_t* empty = full + NB * ST_STAGES;
    StageRec* rec = (StageRec*)(st + ST_STAGES * ST_STAGE_BYTES + (((NB + 1) * ST_STAGES * 8 + 15) & ~15));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < ST_STAGES; ++s) { for (int b = 0; b < NB; ++b) mbar_init(&full[NB * s + b], 1); mbar_init(&empty[s], 1); }
        mbar_init_fence();
    }
    __syncthreads();

    if (warp == 0) {
        // ---- producer: one thread hands boxes to the TMA unit, ST_STAGES boxes (48 KB) ahead of the consumers ----------------
        if (lane != 0) return;
        asm volatile("prefetch.tensormap [%0];" :: "l"(&tmap) : "memory");
        uint64_t policy;
        asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
        const int per_frame = a.TY * a.XB;
        int q = 0;
        int nb = a.item_begin + atomicAdd(a.work, ST_GRAB);
        while (nb < a.item_end) {
            const int base = nb;
            nb = a.item_begin + atomicAdd(a.work, ST_GRAB);                  // the next draw is in flight while this one is posted
            const int end = min(base + ST_GRAB, a.item_end);
            int f = base / per_frame, rem = base - f * per_frame, cy = rem / a.XB, xb = rem - cy * a.XB;
            int chunk = base / a.items_per_chunk, left = (chunk + 1) * a.items_per_chunk - base;
            for (int it = base; it < end; ++it, ++q) {
                const int stage = q % ST_STAGES, fill = q / ST_STAGES;
                uint64_t* fb = &full[NB * stage + fill % NB];
                mbar_wait(&empty[stage], (fill & 1) ^ 1);
                StageRec r;
                r.cb_index = (f * a.TY + cy) * a.TX + xb * (ST_BOX_W / 32); r.ncell = min(ST_BOX_W / 32, a.TX - xb * (ST_BOX_W / 32));
                r.chunk = chunk; r.pad = 0;
                rec[stage] = r;
                mbar_expect_tx(fb, ST_STAGE_BYTES);
                tma_load_box(ring + stage * ST_STAGE_BYTES, &tmap, xb * ST_BOX_W, cy * ST_BOX_H, f, fb, policy);
                if (++xb == a.XB) { xb = 0; if (++cy == a.TY) { cy = 0; ++f; } }
                if (--left == 0) { ++chunk; left = a.items_per_chunk; }
            }
        }
        for (int c = 0; c < ST_CONSUMERS; ++c, ++q) {                        // one end mark per consumer warp
            const int stage = q % ST_STAGES, fill = q / ST_STAGES;
            mbar_wait(&empty[stage], (fill & 1) ^ 1);
            rec[stage].ncell = -1;
            mbar_arrive(&full[NB * stage + fill % NB]);
        }
        return;
    }

    // ---- consumers: warp c takes boxes c, c + ST_CONSUMERS, ...  Lane = (row parity, 16-byte column chunk): 16 loads of 16
    //      bytes cover rows parity, parity + 2, ... of one half cell.  Per lane: the hot bits of its 16 columns OR-ed over the
    //      rows (four words, exact per column) and one bit per hot row. ----------------------------------------------------
    const int cw = warp - 1;
    const int chunkl = lane & 15, rpar = lane >> 4;
    int cur_chunk = -1, cur_cnt = 0;
    for (int q = cw;; q += ST_CONSUMERS) {
        const int stage = q % ST_STAGES, fill = q / ST_STAGES;
        mbar_wait(&full[NB * stage + fill % NB], (fill / NB) & 1);
        const StageRec r = rec[stage];
        if (r.ncell < 0) {                                                   // end mark: hand the slot back (the ring may be shorter than
            __syncwarp();                                                    // the number of consumer warps, the next mark needs a slot)
            if (lane == 0) mbar_arrive(&empty[stage]);
            break;
        }
        const uint8_t* src = ring + stage * ST_STAGE_BYTES + rpar * ST_BOX_W + chunkl * 16;
        uint32_t a0 = 0, a1 = 0, a2 = 0, a3 = 0, rowbits = 0;
        // MODE 0 (thresh >= 128): a hot byte has bit 7 set, so four loads (eight rows) are first OR-ed together -- two LOP3 per load --
        // and the exact per-byte test only runs where some lane of the warp saw such a byte (warp-uniform branch)
#pragma unroll
        for (int k4 = 0; k4 < ST_BOX_H / 2; k4 += 4) {
            uint4 v[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) v[j] = *(const uint4*)(src + (k4 + j) * 2 * ST_BOX_W);
            if (MODE == 0) {
                uint32_t o = 0;
#pragma unroll
                for (int j = 0; j < 4; ++j) o |= v[j].x | v[j].y | v[j].z | v[j].w;
                if (!__any_sync(0xffffffffu, (o & 0x80808080u) != 0)) continue;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t h0 = hot4<MODE>(v[j].x, a.add), h1 = hot4<MODE>(v[j].y, a.add), h2 = hot4<MODE>(v[j].z, a.add), h3 = hot4<MODE>(v[j].w, a.add);
                a0 |= h0; a1 |= h1; a2 |= h2; a3 |= h3;
                if ((h0 | h1 | h2 | h3) & 0x80808080u) rowbits |= 1u << (2 * (k4 + j));
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[stage]);                           // the box is in registers: the slot can be refilled
        const bool hot = ((a0 | a1 | a2 | a3) & 0x80808080u) != 0;
        uint32_t box = CELL_EMPTY;
        if (__ballot_sync(0xffffffffu, hot)) {                               // warp-uniform: some cell of this box is hot
            uint32_t cm = hot_nibble(a0) | (hot_nibble(a1) << 4) | (hot_nibble(a2) << 8) | (hot_nibble(a3) << 12);
            cm <<= (lane & 1) * 16;
            uint32_t rb = rowbits << rpar;
            cm |= __shfl_xor_sync(0xffffffffu, cm, 1); cm |= __shfl_xor_sync(0xffffffffu, cm, 16);
            rb |= __shfl_xor_sync(0xffffffffu, rb, 1); rb |= __shfl_xor_sync(0xffffffffu, rb, 16);
            box = pack_cellbox(cm, rb);                                      // lanes 2c, 2c+1, 2c+16, 2c+17 hold cell c
            box = __shfl_sync(0xffffffffu, box, (2 * lane) & 31);
        }
        if (lane < r.ncell) a.cellbox[r.cb_index + lane] = box;
        if (r.chunk != cur_chunk) { scan_publish(a, cur_chunk, cur_cnt, lane); cur_chunk = r.chunk; cur_cnt = 0; }
        ++cur_cnt;
    }
    scan_publish(a, cur_chunk, cur_cnt, lane);
}

// ---------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
typedef CUresult (*PFN_waitValue32)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);

static void* driver_entry(const char* name)
{
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint(name, &fn, cudaEnableDefault, &qr) != cudaSuccess || qr != cudaDriverEntryPointSuccess) return nullptr;
    return fn;
}

bool frames_tensor_map(CUtensorMap* out, const uint8_t* frames, int n, int H, int W, int64_t fstride, int box_w, int box_h, int l2_promotion)
{
    static PFN_encodeTiled encode = (PFN_encodeTiled)driver_entry("cuTensorMapEncodeTiled");
    if (!encode || n <= 0 || H <= 0 || W <= 0) return false;
    if (W % 16 || fstride % 16 || ((uintptr_t)frames) % 16) return false;    // tensor-map strides are multiples of 16 bytes
    const cuuint64_t gdim[3] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)n};
    const cuuint64_t gstr[2] = {(cuuint64_t)W, (cuuint64_t)fstride};
    const cuuint32_t box[3] = {(cuuint32_t)box_w, (cuuint32_t)box_h, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    return encode(out, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, (void*)frames, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_NONE,
                  l2_promotion >= 256 ? CU_TENSOR_MAP_L2_PROMOTION_L2_256B : l2_promotion >= 128 ? CU_TENSOR_MAP_L2_PROMOTION_L2_128B :
                  l2_promotion >= 64 ? CU_TENSOR_MAP_L2_PROMOTION_L2_64B : CU_TENSOR_MAP_L2_PROMOTION_NONE,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

bool scan_tma_supported(const uint8_t* frames, int n, int H, int W, int64_t fstride, int thresh)
{
    const int T = thresh + 1;
    if (T < 1 || T > 255) return false;                                      // the zero fill of the TMA unit must never read as hot
    if (W % 16 || fstride % 16 || ((uintptr_t)frames) % 16) return false;    // tensor-map strides are multiples of 16 bytes
    if (n <= 0 || H <= 0 || W <= 0) return false;
    static const bool have = driver_entry("cuTensorMapEncodeTiled") != nullptr;
    return have;
}

// One launch over every box of the batch.  ctrl: the control block, zeroed by the caller on an earlier point of the stream.
int launch_scan_tma(const uint8_t* frames, int n, int H, int W, int64_t fstride, const TableView& tv, int thresh, uint32_t* cellbox,
                    int* ctrl, int chunks, int chunk_frames, cudaStream_t s)
{
    CUtensorMap map;
    if (!frames_tensor_map(&map, frames, n, H, W, fstride, ST_BOX_W, ST_BOX_H, 256)) return MOCAP_ERR_UNSUPPORTED;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const HotTest ht = make_hot_test(thresh);
    ScanTmaArgs a;
    a.cellbox = cellbox;
    a.work = ctrl;
    a.chunk_done = ctrl + SCAN_CTRL_WORK;
    a.chunk_flag = ctrl + SCAN_CTRL_WORK + chunks;
    a.TX = tv.TX; a.TY = tv.TY; a.XB = cdiv(W, ST_BOX_W);
    const long long per_frame = (long long)a.TY * a.XB;
    if (per_frame * n >= (1LL << 31) - 64 * ST_GRAB * sms) return MOCAP_ERR_UNSUPPORTED;
    a.total_items = (int)(per_frame * n);
    a.items_per_chunk = (int)(per_frame * chunk_frames);
    a.item_begin = 0; a.item_end = a.total_items;
    a.add = ht.add;
    const int smem = ST_STAGES * ST_STAGE_BYTES + 4 * ST_STAGES * 8 + 16 + ST_STAGES * (int)sizeof(StageRec) + 128;
    static bool attr_done = false;
    if (!attr_done) {
        CUDA_TRY(cudaFuncSetAttribute(scan_tma_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        CUDA_TRY(cudaFuncSetAttribute(scan_tma_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        attr_done = true;
    }
    mocap_count_launch();
    if (ht.mode == 0) scan_tma_kernel<0><<<sms, ST_THREADS, smem, s>>>(map, a);
    else scan_tma_kernel<1><<<sms, ST_THREADS, smem, s>>>(map, a);
    CUDA_TRY(cudaGetLastError());
    return MOCAP_OK;
}

// stream `s` continues once the 32-bit word at `addr_dev` is >= value (cuStreamWaitValue32: no SM is held while waiting)
int stream_wait_geq(cudaStream_t s, const int* addr_dev, int value)
{
    static PFN_waitValue32 wait = (PFN_waitValue32)driver_entry("cuStreamWaitValue32");
    if (!wait) return MOCAP_ERR_UNSUPPORTED;
    return wait((CUstream)s, (CUdeviceptr)(uintptr_t)addr_dev, (cuuint32_t)value, CU_STREAM_WAIT_VALUE_GEQ) == CUDA_SUCCESS ? MOCAP_OK : MOCAP_ERR_CUDA;
}
bool stream_wait_supported()
{
    static const bool have = driver_entry("cuStreamWaitValue32") != nullptr;
    return have;
}

#else   // MOCAP_EMU: the CPU emulation build of the kernel sources (tests/emu) runs no TMA scan; the classic scan kernels serve there

// the stand-in tensor map of the emulation build (tma.cuh), for the same batches the driver describes above
bool frames_tensor_map(CUtensorMap* out, const uint8_t* frames, int n, int H, int W, int64_t fstride, int box_w, int box_h, int)
{
    if (n <= 0 || H <= 0 || W <= 0) return false;
    if (W % 16 || fstride % 16 || ((uintptr_t)frames) % 16) return false;    // tensor-map strides are multiples of 16 bytes
    *out = CUtensorMap{frames, n, H, W, fstride, box_w, box_h};
    return true;
}
bool scan_tma_supported(const uint8_t*, int, int, int, int64_t, int) { return false; }
int launch_scan_tma(const uint8_t*, int, int, int, int64_t, const TableView&, int, uint32_t*, int*, int, int, cudaStream_t) { return MOCAP_ERR_UNSUPPORTED; }
int stream_wait_geq(cudaStream_t, const int*, int) { return MOCAP_ERR_UNSUPPORTED; }
bool stream_wait_supported() { return false; }

#endif
