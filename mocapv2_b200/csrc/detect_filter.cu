// Detection front end: frames (u8, HBM) -> filtered binary image (bit-packed) for _find_dot.
//
// Replaces, for a batch of frames, lib/ImageOperations.py:38-40 of the reference:
//     cv.undistort(img, K0, dist0) -> fast_cuda_blur(.,5) -> cv.threshold(.,216.75) -> cv.medianBlur(.,5)
// with the exact integer semantics pinned in oracle/restate.py (SURVEY.md App. A1-A4).
//
// Design (sparse, HBM-bound):
//   scan_hot      streams every source byte once (16-byte loads) and marks the output tiles that a source
//                 cell holding a pixel > thresh can influence.  A filtered pixel can only be set if some
//                 source tap within reach is > thresh (bilinear weights sum to 1, box mean <= max), so
//                 unmarked tiles are exactly zero and are never touched again.
//   compact       turns the per-frame active-tile bitmaps into a work list.
//   filter_tiles  one warp per active 32x32 tile: exact hot bounding box of the tile's source window,
//                 fixed-point remap + 5x5 floor-mean threshold + 5x5 majority only inside that box.
#include "common.cuh"
#include "remap.cuh"

// ---------------------------------------------------------------------------------------------------------
// table build
// ---------------------------------------------------------------------------------------------------------
struct MapParams {
    double ir[9];
    double fx, fy, cx, cy, k1, k2, p1, p2, k3;
};

// FP64 map of cv::initUndistortRectifyMap(K, dist, I, K), same operation order as oracle.restate
// (no FMA contraction: every product and sum is rounded separately).
__global__ void build_map_kernel(MapParams mp, int H, int W, int32_t* __restrict__ map, TableHeader* hdr)
{
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    int i = blockIdx.y * blockDim.y + threadIdx.y;
    if (i >= H || j >= W) return;
    double di = (double)i, dj = (double)j;
    double _x = __dadd_rn(__dadd_rn(__dmul_rn(di, mp.ir[1]), mp.ir[2]), __dmul_rn(dj, mp.ir[0]));
    double _y = __dadd_rn(__dadd_rn(__dmul_rn(di, mp.ir[4]), mp.ir[5]), __dmul_rn(dj, mp.ir[3]));
    double _w = __dadd_rn(__dadd_rn(__dmul_rn(di, mp.ir[7]), mp.ir[8]), __dmul_rn(dj, mp.ir[6]));
    double w = __ddiv_rn(1.0, _w);
    double x = __dmul_rn(_x, w), y = __dmul_rn(_y, w);
    double x2 = __dmul_rn(x, x), y2 = __dmul_rn(y, y);
    double r2 = __dadd_rn(x2, y2);
    double _2xy = __dmul_rn(__dmul_rn(2.0, x), y);
    double kr = __dadd_rn(1.0, __dmul_rn(__dadd_rn(__dmul_rn(__dadd_rn(__dmul_rn(mp.k3, r2), mp.k2), r2), mp.k1), r2));
    double xd = __dadd_rn(__dadd_rn(__dmul_rn(x, kr), __dmul_rn(mp.p1, _2xy)),
                          __dmul_rn(mp.p2, __dadd_rn(r2, __dmul_rn(2.0, x2))));
    double yd = __dadd_rn(__dadd_rn(__dmul_rn(y, kr), __dmul_rn(mp.p1, __dadd_rn(r2, __dmul_rn(2.0, y2)))),
                          __dmul_rn(mp.p2, _2xy));
    double u = __dadd_rn(__dmul_rn(mp.fx, xd), mp.cx);
    double v = __dadd_rn(__dmul_rn(mp.fy, yd), mp.cy);
    double u32 = __dmul_rn(u, 32.0), v32 = __dmul_rn(v, 32.0);
    uint32_t enc = MAP_OUTSIDE;
    if (fabs(u32) < 1.0e9 && fabs(v32) < 1.0e9) {          // also rejects NaN
        long long iu = __double2ll_rn(u32), iv = __double2ll_rn(v32);   // rint (ties to even) like cvRound
        long long sx = iu >> 5, sy = iv >> 5;
        if (sx >= -1 && sx <= W - 1 && sy >= -1 && sy <= H - 1) {
            long long du = iu - 32LL * j, dv = iv - 32LL * i;
            if (du > -32768 && du < 32768 && dv > -32768 && dv < 32768)
                enc = ((uint32_t)(du & 0xffff)) | ((uint32_t)(dv & 0xffff) << 16);
            else
                atomicAdd(&hdr->overflow, 1);
        }
    }
    if (enc == MAP_OUTSIDE) atomicAdd(&hdr->n_zero, 1);
    map[(size_t)i * W + j] = (int32_t)enc;
}

__global__ void init_tables_kernel(int32_t* cell, int32_t* tile, int32_t* cellinv, int n_tiles)
{
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tiles) return;
    cell[4 * t + 0] = 0x7fffffff; cell[4 * t + 1] = 0x7fffffff; cell[4 * t + 2] = -1; cell[4 * t + 3] = -1;
    cellinv[4 * t + 0] = 0x7fffffff; cellinv[4 * t + 1] = -0x7fffffff; cellinv[4 * t + 2] = 0x7fffffff; cellinv[4 * t + 3] = -0x7fffffff;
}

// one CTA per output tile: source window + displacement bounds of its 40x40 undistorted region,
// then scatter the tile index into the reach rectangle of every source cell the window overlaps.
__global__ void build_tile_kernel(const int32_t* __restrict__ map, int H, int W, int TX, int TY,
                                  int32_t* __restrict__ cell, int32_t* __restrict__ tile, int32_t* __restrict__ cellinv)
{
    int tx = blockIdx.x, ty = blockIdx.y;
    int x0 = tx * TILE - HALO_U, y0 = ty * TILE - HALO_U;
    __shared__ int s[8];
    if (threadIdx.x < 8) s[threadIdx.x] = (threadIdx.x & 1) ? -0x7fffffff : 0x7fffffff;   // even: min, odd: max
    __syncthreads();
    int mn[4] = {0x7fffffff, 0x7fffffff, 0x7fffffff, 0x7fffffff};
    int mx[4] = {-0x7fffffff, -0x7fffffff, -0x7fffffff, -0x7fffffff};
    for (int idx = threadIdx.x; idx < REG_U * REG_U; idx += blockDim.x) {
        int i = y0 + idx / REG_U, j = x0 + idx % REG_U;
        if (i < 0 || j < 0 || i >= H || j >= W) continue;
        uint32_t m = (uint32_t)map[(size_t)i * W + j];
        if (m == MAP_OUTSIDE) continue;
        int du = (int16_t)(m & 0xffff), dv = (int16_t)(m >> 16);
        int ddx = du >> 5, ddy = dv >> 5;          // integer displacement (floor)
        int sx = j + ddx, sy = i + ddy;
        mn[0] = min(mn[0], sx); mx[0] = max(mx[0], sx + 1);
        mn[1] = min(mn[1], sy); mx[1] = max(mx[1], sy + 1);
        mn[2] = min(mn[2], ddx); mx[2] = max(mx[2], ddx);
        mn[3] = min(mn[3], ddy); mx[3] = max(mx[3], ddy);
    }
    for (int k = 0; k < 4; ++k) { atomicMin(&s[2 * k], mn[k]); atomicMax(&s[2 * k + 1], mx[k]); }
    __syncthreads();
    if (threadIdx.x == 0) {
        int32_t* t = tile + 8 * (ty * TX + tx);
        int sx0 = max(s[0], 0), sx1 = min(s[1], W - 1), sy0 = max(s[2], 0), sy1 = min(s[3], H - 1);
        if (s[0] == 0x7fffffff) { sx0 = 0; sx1 = -1; sy0 = 0; sy1 = -1; }
        t[0] = sx0; t[1] = sy0; t[2] = sx1; t[3] = sy1;
        t[4] = s[4]; t[5] = s[5]; t[6] = s[6]; t[7] = s[7];
        for (int cy = sy0 >> 5; cy <= (sy1 >> 5); ++cy)
            for (int cx = sx0 >> 5; cx <= (sx1 >> 5); ++cx) {
                int32_t* c = cell + 4 * (cy * TX + cx);
                atomicMin(&c[0], tx); atomicMin(&c[1], ty); atomicMax(&c[2], tx); atomicMax(&c[3], ty);
            }
    }
}

// The map in the form the piece filter's fast path consumes (TableHeader::off_fast) + per output tile whether all of its pixels have one.
// One CTA per output tile.
__global__ void build_fast_kernel(const int32_t* __restrict__ map, int H, int W, int TX, int32_t* __restrict__ fast, int32_t* __restrict__ tflag)
{
    const int tx = blockIdx.x, ty = blockIdx.y;
    __shared__ int s_bad;
    if (threadIdx.x == 0) s_bad = 0;
    __syncthreads();
    int bad = 0;
    for (int idx = threadIdx.x; idx < TILE * TILE; idx += blockDim.x) {
        int i = ty * TILE + idx / TILE, j = tx * TILE + idx % TILE;
        if (i >= H || j >= W) continue;
        uint32_t m = (uint32_t)map[(size_t)i * W + j], enc = FAST_INVALID;
        if (m != MAP_OUTSIDE) {
            int du = (int16_t)(m & 0xffff), dv = (int16_t)(m >> 16);
            int off = (dv >> 5) * WIN_W + (du >> 5);
            if (off >= -32768 && off <= 32767) enc = (uint32_t)(du & 31) | ((uint32_t)(dv & 31) << 8) | ((uint32_t)off << 16);
        }
        if (enc == FAST_INVALID) bad = 1;
        fast[(size_t)i * W + j] = (int32_t)enc;
    }
    if (tx == 0 && ty == 0 && threadIdx.x < 4) fast[(size_t)H * W + threadIdx.x] = 0;      // the pad behind the last row
    if (bad) atomicOr(&s_bad, 1);
    __syncthreads();
    if (threadIdx.x == 0) tflag[ty * TX + tx] = s_bad;
}

// Per 32x32 source cell: exact bounds of (source - output) integer displacement over every output pixel whose 2x2 tap
// footprint touches the cell.  One thread per output pixel; pixels of a warp mostly hit the same cell, so the atomics are
// few per address and this runs once per calibration.
__global__ void build_cellinv_kernel(const int32_t* __restrict__ map, int H, int W, int TX, int32_t* __restrict__ cellinv)
{
    int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y * blockDim.y + threadIdx.y;
    if (i >= H || j >= W) return;
    uint32_t m = (uint32_t)map[(size_t)i * W + j];
    if (m == MAP_OUTSIDE) return;
    int ddx = (int)(int16_t)(m & 0xffff) >> 5, ddy = (int)(int16_t)(m >> 16) >> 5;
    int sx = j + ddx, sy = i + ddy;
    for (int ty = 0; ty < 2; ++ty)
        for (int tx = 0; tx < 2; ++tx) {
            int x = sx + tx, y = sy + ty;
            if ((unsigned)x >= (unsigned)W || (unsigned)y >= (unsigned)H) continue;
            if ((tx && ((x & 31) != 0)) || (ty && ((y & 31) != 0))) continue;      // same cell as the tap before it
            int32_t* ci = cellinv + 4 * ((y >> 5) * TX + (x >> 5));
            if (ci[0] > ddx) atomicMin(&ci[0], ddx);
            if (ci[1] < ddx) atomicMax(&ci[1], ddx);
            if (ci[2] > ddy) atomicMin(&ci[2], ddy);
            if (ci[3] < ddy) atomicMax(&ci[3], ddy);
        }
}

static void invert3x3(const double* A, double* out)
{
    // closed-form adjugate inverse (what cv::invert does for 3x3): cofactors times 1/det
    double d = A[0] * (A[4] * A[8] - A[5] * A[7]) - A[1] * (A[3] * A[8] - A[5] * A[6]) + A[2] * (A[3] * A[7] - A[4] * A[6]);
    d = 1.0 / d;
    out[0] = (A[4] * A[8] - A[5] * A[7]) * d;
    out[1] = (A[2] * A[7] - A[1] * A[8]) * d;
    out[2] = (A[1] * A[5] - A[2] * A[4]) * d;
    out[3] = (A[5] * A[6] - A[3] * A[8]) * d;
    out[4] = (A[0] * A[8] - A[2] * A[6]) * d;
    out[5] = (A[2] * A[3] - A[0] * A[5]) * d;
    out[6] = (A[3] * A[7] - A[4] * A[6]) * d;
    out[7] = (A[1] * A[6] - A[0] * A[7]) * d;
    out[8] = (A[0] * A[4] - A[1] * A[3]) * d;
}

static void table_layout(int H, int W, TableHeader* h)
{
    h->magic = TABLE_MAGIC;
    h->H = H; h->W = W;
    h->TX = cdiv(W, TILE); h->TY = cdiv(H, TILE);
    h->overflow = 0; h->n_zero = 0; h->pad = 0;
    size_t off = align_up(sizeof(TableHeader), 256);
    h->off_map = off; off += align_up((size_t)H * W * 4, 256);
    h->off_cell = off; off += align_up((size_t)h->TX * h->TY * 16, 256);
    h->off_tile = off; off += align_up((size_t)h->TX * h->TY * 32, 256);
    h->off_cellinv = off; off += align_up((size_t)h->TX * h->TY * 16, 256);
    h->off_fast = off; off += align_up((size_t)H * W * 4 + 16, 256);
    h->off_tflag = off; off += align_up((size_t)h->TX * h->TY * 4, 256);
    h->total_bytes = off;
}

extern "C" size_t mocap_undistort_table_bytes(int H, int W)
{
    if (H <= 0 || W <= 0) return 0;
    TableHeader h; table_layout(H, W, &h);
    return (size_t)h.total_bytes;
}

extern "C" int mocap_undistort_table_build(const double* K9, const double* dist5, int H, int W,
                                           void* table_dev, size_t table_bytes, void* stream)
{
    if (!K9 || !dist5 || !table_dev || H <= 0 || W <= 0) return MOCAP_ERR_INVALID;
    if (H > 16384 || W > 16384) return MOCAP_ERR_UNSUPPORTED;
    TableHeader h; table_layout(H, W, &h);
    if (table_bytes < h.total_bytes) return MOCAP_ERR_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    MapParams mp;
    invert3x3(K9, mp.ir);
    mp.fx = K9[0]; mp.fy = K9[4]; mp.cx = K9[2]; mp.cy = K9[5];
    mp.k1 = dist5[0]; mp.k2 = dist5[1]; mp.p1 = dist5[2]; mp.p2 = dist5[3]; mp.k3 = dist5[4];
    char* base = (char*)table_dev;
    CUDA_TRY(cudaMemcpyAsync(base, &h, sizeof(h), cudaMemcpyHostToDevice, s));
    int32_t* map = (int32_t*)(base + h.off_map);
    int32_t* cell = (int32_t*)(base + h.off_cell);
    int32_t* tile = (int32_t*)(base + h.off_tile);
    int32_t* cellinv = (int32_t*)(base + h.off_cellinv);
    dim3 blk(32, 8), grd(cdiv(W, 32), cdiv(H, 8));
    LAUNCH(build_map_kernel, grd, blk, 0, s, mp, H, W, map, (TableHeader*)base);
    int nt = h.TX * h.TY;
    LAUNCH(init_tables_kernel, cdiv(nt, 256), 256, 0, s, cell, tile, cellinv, nt);
    LAUNCH(build_tile_kernel, dim3(h.TX, h.TY), 256, 0, s, map, H, W, h.TX, h.TY, cell, tile, cellinv);
    LAUNCH(build_cellinv_kernel, grd, blk, 0, s, map, H, W, h.TX, cellinv);
    LAUNCH(build_fast_kernel, dim3(h.TX, h.TY), 256, 0, s, map, H, W, h.TX, (int32_t*)(base + h.off_fast), (int32_t*)(base + h.off_tflag));
    CUDA_TRY(cudaGetLastError());
    TableHeader back;
    CUDA_TRY(cudaMemcpyAsync(&back, base, sizeof(back), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    if (back.overflow) return MOCAP_ERR_UNSUPPORTED;   // displacement beyond +-1023 px
    return MOCAP_OK;
}

int table_view(const void* table_dev, int H, int W, TableView* tv)
{
    // layout is a pure function of (H, W); the header on the device is only read by kernels
    TableHeader h; table_layout(H, W, &h);
    const char* base = (const char*)table_dev;
    tv->map = (const int32_t*)(base + h.off_map);
    tv->cell = (const int32_t*)(base + h.off_cell);
    tv->tile = (const int32_t*)(base + h.off_tile);
    tv->cellinv = (const int32_t*)(base + h.off_cellinv);
    tv->fast = (const int32_t*)(base + h.off_fast);
    tv->tflag = (const int32_t*)(base + h.off_tflag);
    tv->H = H; tv->W = W; tv->TX = h.TX; tv->TY = h.TY;
    tv->lens_words = 0; tv->n_lenses = 1; tv->frame_lens = nullptr;
    return MOCAP_OK;
}

__device__ __forceinline__ uint4 ldg_stream16(const void* p)
{
#ifdef MOCAP_EMU
    return *(const uint4*)p;
#else
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::128B.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
#endif
}

__device__ __forceinline__ void mark_cell(const TableView& tv, uint32_t* __restrict__ active, int f, int cy, int cx, int TXW)
{
    const int32_t* c = tv.cell + 4 * (cy * tv.TX + cx);
    int tx0 = c[0], ty0 = c[1], tx1 = c[2], ty1 = c[3];
    if (tx1 < tx0) return;
    for (int ty = ty0; ty <= ty1; ++ty) {
        uint32_t* row = active + ((size_t)f * tv.TY + ty) * TXW;
        for (int wq = tx0 >> 5; wq <= (tx1 >> 5); ++wq) {
            int lo = max(tx0, wq * 32) - wq * 32, hi = min(tx1, wq * 32 + 31) - wq * 32;
            uint32_t m = (hi == 31 ? 0xffffffffu : ((1u << (hi + 1)) - 1u)) & ~((1u << lo) - 1u);
            if ((row[wq] & m) != m) atomicOr(&row[wq], m);
        }
    }
}

// Streams all source bytes.  One warp per 128x32-pixel block (4 source cells): lane = (row & 3, 16-byte segment).
// Writes the hot bounding box of every cell (cellbox); that is all later stages need to know about the frame.
template <int MODE>
__global__ void __launch_bounds__(256, 4) scan_hot_vec_kernel(const uint8_t* __restrict__ frames, int n_frames, int64_t fstride,
                                                              TableView tv, uint32_t add, uint32_t* __restrict__ cellbox)
{
    const int lane = threadIdx.x & 31;
    const unsigned warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const unsigned nwarps = (gridDim.x * blockDim.x) >> 5;
    const int H = tv.H, W = tv.W;
    const unsigned CXB = (unsigned)(tv.TX + 3) >> 2;
    const unsigned per_frame = (unsigned)tv.TY * CXB;
    const unsigned total = per_frame * (unsigned)n_frames;         // < 2^31: the work-list codes of the library are 32-bit anyway
    const int seg = lane & 7, r0 = lane >> 3;
    for (unsigned it = warp; it < total; it += nwarps) {
        int f = (int)(it / per_frame);
        int rem = (int)(it - (unsigned)f * per_frame);
        int cy = rem / (int)CXB, cxb = rem - cy * (int)CXB;
        int x = cxb * 128 + seg * 16;
        const uint8_t* base = frames + (size_t)f * fstride + (size_t)(cy * 32 + r0) * W + x;
        bool colok = x < W;
        uint32_t acc = 0;
        uint4 v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            int row = cy * 32 + k * 4 + r0;
            if (colok && row < H) v[k] = ldg_stream16(base + (size_t)(k * 4) * W);
            else v[k] = make_uint4(0, 0, 0, 0);
        }
#pragma unroll
        for (int k = 0; k < 8; ++k)
            acc |= hot4<MODE>(v[k].x, add) | hot4<MODE>(v[k].y, add) | hot4<MODE>(v[k].z, add) | hot4<MODE>(v[k].w, add);
        bool hot = (acc & 0x80808080u) != 0;
        unsigned m = __ballot_sync(0xffffffffu, hot);
        uint32_t box = CELL_EMPTY;
        if (m) {                                            // warp-uniform: some cell of this block is hot
            uint32_t colmask = 0, rowbits = 0;              // lane-local: hot columns (16 bits), hot rows (bit 4k + r0)
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                uint32_t c = hot_nibble(hot4<MODE>(v[k].x, add)) | (hot_nibble(hot4<MODE>(v[k].y, add)) << 4) |
                             (hot_nibble(hot4<MODE>(v[k].z, add)) << 8) | (hot_nibble(hot4<MODE>(v[k].w, add)) << 12);
                colmask |= c;
                if (c) rowbits |= 1u << (4 * k + r0);
            }
            colmask <<= (seg & 1) * 16;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                bool mine = (seg >> 1) == c;
                uint32_t xm = __reduce_or_sync(0xffffffffu, mine ? colmask : 0u);
                uint32_t ym = __reduce_or_sync(0xffffffffu, mine ? rowbits : 0u);
                if (lane == c) box = pack_cellbox(xm, ym);
            }
        }
        if (lane < 4) {
            int cx = cxb * 4 + lane;
            if (cx < tv.TX) cellbox[((size_t)f * tv.TY + cy) * tv.TX + cx] = box;
        }
    }
}

// 32 bytes per lane with one 256-bit load (sm_100: LDG.E.256) that also carries the L2 evict-first priority: the frames
// are read exactly once per batch, so they should not push the undistortion map and the clusters' bit rows out of L2.
struct uint8w { uint32_t w[8]; };
__device__ __forceinline__ uint8w ldg_stream32(const void* p)
{
    uint8w r;
#ifdef MOCAP_EMU
    memcpy(&r, p, 32);
#else
    asm volatile("ld.global.nc.L1::no_allocate.L2::evict_first.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r.w[0]), "=r"(r.w[1]), "=r"(r.w[2]), "=r"(r.w[3]), "=r"(r.w[4]), "=r"(r.w[5]), "=r"(r.w[6]), "=r"(r.w[7]) : "l"(p));
#endif
    return r;
}

// Same as scan_hot_vec_kernel for rows that are 32-byte aligned: lane = (row & 7, 32-byte segment = one source cell)
template <int MODE>
__global__ void __launch_bounds__(256, 4) scan_hot_vec32_kernel(const uint8_t* __restrict__ frames, int n_frames, int64_t fstride,
                                                                TableView tv, uint32_t add, uint32_t* __restrict__ cellbox)
{
    const int lane = threadIdx.x & 31;
    const unsigned warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const unsigned nwarps = (gridDim.x * blockDim.x) >> 5;
    const int H = tv.H, W = tv.W;
    const unsigned CXB = (unsigned)(tv.TX + 3) >> 2;
    const unsigned per_frame = (unsigned)tv.TY * CXB;
    const unsigned total = per_frame * (unsigned)n_frames;
    const int seg = lane & 3, r0 = lane >> 2;
    for (unsigned it = warp; it < total; it += nwarps) {
        int f = (int)(it / per_frame);
        int rem = (int)(it - (unsigned)f * per_frame);
        int cy = rem / (int)CXB, cxb = rem - cy * (int)CXB;
        int x = cxb * 128 + seg * 32;
        const uint8_t* base = frames + (size_t)f * fstride + (size_t)(cy * 32 + r0) * W + x;
        bool colok = x < W;
        uint32_t acc = 0;
        uint8w v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            int row = cy * 32 + k * 8 + r0;
            if (colok && row < H) v[k] = ldg_stream32(base + (size_t)(k * 8) * W);
            else {
#pragma unroll
                for (int q = 0; q < 8; ++q) v[k].w[q] = 0;
            }
        }
#pragma unroll
        for (int k = 0; k < 4; ++k)
#pragma unroll
            for (int q = 0; q < 8; ++q) acc |= hot4<MODE>(v[k].w[q], add);
        bool hot = (acc & 0x80808080u) != 0;
        unsigned m = __ballot_sync(0xffffffffu, hot);
        uint32_t box = CELL_EMPTY;
        if (m) {                                            // warp-uniform: some cell of this block is hot
            uint32_t colmask = 0, rowbits = 0;              // lane-local: hot columns of the cell (32 bits), hot rows (bit 8k + r0)
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                uint32_t c = 0;
#pragma unroll
                for (int q = 0; q < 8; ++q) c |= hot_nibble(hot4<MODE>(v[k].w[q], add)) << (4 * q);
                colmask |= c;
                if (c) rowbits |= 1u << (8 * k + r0);
            }
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                bool mine = seg == c;
                uint32_t xm = __reduce_or_sync(0xffffffffu, mine ? colmask : 0u);
                uint32_t ym = __reduce_or_sync(0xffffffffu, mine ? rowbits : 0u);
                if (lane == c) box = pack_cellbox(xm, ym);
            }
        }
        if (lane < 4) {
            int cx = cxb * 4 + lane;
            if (cx < tv.TX) cellbox[((size_t)f * tv.TY + cy) * tv.TX + cx] = box;
        }
    }
}

// Generic (any W / alignment) variant: one warp per source cell, byte loads.
__global__ void scan_hot_scalar_kernel(const uint8_t* __restrict__ frames, int n_frames, int64_t fstride,
                                       TableView tv, int thresh, uint32_t* __restrict__ cellbox)
{
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const int H = tv.H, W = tv.W;
    const long long per_frame = (long long)tv.TY * tv.TX;
    const long long total = per_frame * n_frames;
    for (long long it = warp; it < total; it += nwarps) {
        int f = (int)(it / per_frame);
        int rem = (int)(it - (long long)f * per_frame);
        int cy = rem / tv.TX, cx = rem - cy * tv.TX;
        int x = cx * 32 + lane;
        uint32_t rowbits = 0;
        if (x < W) {
            const uint8_t* base = frames + (size_t)f * fstride + x;
            for (int r = 0; r < 32; ++r) {
                int y = cy * 32 + r;
                if (y < H && (int)base[(size_t)y * W] > thresh) rowbits |= 1u << r;
            }
        }
        uint32_t xm = __ballot_sync(0xffffffffu, rowbits != 0);
        uint32_t ym = __reduce_or_sync(0xffffffffu, rowbits);
        if (lane == 0) cellbox[((size_t)f * tv.TY + cy) * tv.TX + cx] = pack_cellbox(xm, ym);
    }
}

// general path: the output tiles the hot cells of a flagged frame can reach (one CTA per frame; frames the cluster path
// finished leave at once).  A frame whose lens index is out of range marks no tile: nothing downstream reads a table for it.
__global__ void mark_active_kernel(const uint32_t* __restrict__ cellbox, TableView tv, int n_frames, uint32_t* __restrict__ active, int TXW,
                                   const int* __restrict__ need_general, int* __restrict__ flags)
{
    const int cells = tv.TX * tv.TY;
    for (int f = blockIdx.x; f < n_frames; f += gridDim.x) {
        if (need_general && !need_general[f]) continue;
        const int lens = frame_lens_of(tv, f);
        if (lens < 0) { if (threadIdx.x == 0) flags[f] |= MOCAP_FLAG_LENS_INDEX; continue; }
        const TableView tl = lens_table(tv, lens);
        const uint32_t* cb = cellbox + (size_t)f * cells;
        for (int c = threadIdx.x; c < cells; c += blockDim.x)
            if (cb[c] != CELL_EMPTY) mark_cell(tl, active, f, c / tv.TX, c % tv.TX, TXW);
    }
}

__global__ void compact_tiles_kernel(const uint32_t* __restrict__ active, long long n_words, int TX, int TY, int TXW,
                                     uint32_t* __restrict__ list, int* __restrict__ count, const int* __restrict__ need_general)
{
    long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n_words) return;
    uint32_t w = active[idx];
    if (!w) return;
    int f = (int)(idx / ((long long)TY * TXW));
    if (need_general && !need_general[f]) return;          // frame fully handled by the cluster path
    int rem = (int)(idx - (long long)f * TY * TXW);
    int ty = rem / TXW, wq = rem - ty * TXW;
    int base = atomicAdd(count, __popc(w));
    while (w) {
        int b = __ffs(w) - 1;
        w &= w - 1;
        list[base++] = (uint32_t)f * (uint32_t)(TX * TY) + (uint32_t)(ty * TX + wq * 32 + b);
    }
}

// ---------------------------------------------------------------------------------------------------------
// filter_tiles: one warp per active tile
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int fdiv20(int idx, int inv) { return (int)(((unsigned)idx * (unsigned)inv) >> 20); }
__device__ __forceinline__ int finv20(int w) { return (1 << 20) / w + 1; }

#define FT_WARPS 8
struct __align__(16) WarpScratch {
    uint8_t U[REG_U * REG_U];        // undistorted pixels, origin (x0-4, y0-4)
    uint16_t HS[REG_U * REG_B];      // horizontal 5-sums of U: rows = U rows, cols = B cols; reused for majority sums
    uint8_t B[REG_B * REG_B];        // thresholded box mean, origin (x0-2, y0-2)
};

__global__ void __launch_bounds__(FT_WARPS * 32) filter_tiles_kernel(
    const uint8_t* __restrict__ frames, int64_t fstride, TableView tv, int thresh,
    const uint32_t* __restrict__ list, const int* __restrict__ n_list, int* __restrict__ cursor,
    const uint32_t* __restrict__ active, int TXW, const uint32_t* __restrict__ cellbox,
    uint32_t* __restrict__ bits, uint32_t* __restrict__ fg_tiles, int* __restrict__ n_fg, int max_fg, int* __restrict__ flags)
{
    __shared__ WarpScratch scratch[FT_WARPS];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    WarpScratch& S = scratch[wid];
    const int H = tv.H, W = tv.W, TX = tv.TX, TY = tv.TY;
    const int T = thresh + 1;
    const int total = *n_list;
    for (;;) {
        int item = 0;
        if (lane == 0) item = atomicAdd(cursor, 1);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (item >= total) break;
        uint32_t code = list[item];
        int f = (int)(code / (uint32_t)(TX * TY)), t = (int)(code - (uint32_t)f * (uint32_t)(TX * TY));
        int ty = t / TX, tx = t - ty * TX;
        int x0 = tx * TILE, y0 = ty * TILE;
        const uint8_t* fr = frames + (size_t)f * fstride;
        uint32_t* brow = bits + ((size_t)f * H + y0) * TX + tx;
        const size_t loff = tv.frame_lens ? (size_t)tv.frame_lens[f] * tv.lens_words : 0;     // (checked by mark_active_kernel)
        const int32_t* tt = tv.tile + loff + 8 * t;
        const int32_t* map = tv.map + loff;
        int sx0 = tt[0], sy0 = tt[1], sx1 = tt[2], sy1 = tt[3];
        uint32_t myword = 0;

        // ---- 1. hot bounding box of the source window from the scan pass' cell boxes (no pixel is re-read) -------------
        int hx0 = 0x7fffffff, hx1 = -1, hy0 = 0x7fffffff, hy1 = -1;
        if (sx1 >= sx0) {
            int cx0 = sx0 >> 5, cy0 = sy0 >> 5, ncx = (sx1 >> 5) - cx0 + 1, ncy = (sy1 >> 5) - cy0 + 1;
            for (int ci = lane; ci < ncx * ncy; ci += 32) {
                int cy = cy0 + ci / ncx, cx = cx0 + ci % ncx;
                uint32_t b = cellbox[((size_t)f * TY + cy) * TX + cx];
                if (b != CELL_EMPTY) {
                    int bx0 = max(cx * 32 + (int)(b & 0xff), sx0), bx1 = min(cx * 32 + (int)((b >> 8) & 0xff), sx1);
                    int by0 = max(cy * 32 + (int)((b >> 16) & 0xff), sy0), by1 = min(cy * 32 + (int)(b >> 24), sy1);
                    if (bx0 <= bx1 && by0 <= by1) {
                        hx0 = min(hx0, bx0); hx1 = max(hx1, bx1); hy0 = min(hy0, by0); hy1 = max(hy1, by1);
                    }
                }
            }
        }
        hx0 = __reduce_min_sync(0xffffffffu, hx0); hx1 = __reduce_max_sync(0xffffffffu, hx1);
        hy0 = __reduce_min_sync(0xffffffffu, hy0); hy1 = __reduce_max_sync(0xffffffffu, hy1);
        bool any = hx1 >= 0;
        int MX0 = 0, MX1 = -1, MY0 = 0, MY1 = -1;
        if (any) {
            // undistorted pixels that can be > thresh: j in [hx0-1-dxmax, hx1-dxmin], same for rows
            int ux0 = hx0 - 1 - tt[5], ux1 = hx1 - tt[4], uy0 = hy0 - 1 - tt[7], uy1 = hy1 - tt[6];
            // box-mean threshold can fire within +-2 of those, the majority within +-4
            MX0 = max(max(ux0 - 4, x0), 0); MX1 = min(min(ux1 + 4, x0 + TILE - 1), W - 1);
            MY0 = max(max(uy0 - 4, y0), 0); MY1 = min(min(uy1 + 4, y0 + TILE - 1), H - 1);
            any = MX1 >= MX0 && MY1 >= MY0;
            if (any) {
                // B compute box (where the threshold can fire), clipped to the majority's read set
                int BX0 = max(max(ux0 - 2, MX0 - 2), 0), BX1 = min(min(ux1 + 2, MX1 + 2), W - 1);
                int BY0 = max(max(uy0 - 2, MY0 - 2), 0), BY1 = min(min(uy1 + 2, MY1 + 2), H - 1);
                // B read set of the majority (replicated border = clamped coordinates)
                int RX0 = max(MX0 - 2, 0), RX1 = min(MX1 + 2, W - 1), RY0 = max(MY0 - 2, 0), RY1 = min(MY1 + 2, H - 1);
                if (BX1 >= BX0 && BY1 >= BY0) {
                    // ---- 2. U on the B box dilated by 2 (zero outside the frame) ------------------------
                    int UX0 = BX0 - 2, UX1 = BX1 + 2, UY0 = BY0 - 2, UY1 = BY1 + 2;
                    {
                        int bw = UX1 - UX0 + 1, n = bw * (UY1 - UY0 + 1), inv = finv20(bw);
                        for (int idx = lane; idx < n; idx += 32) {
                            int r = fdiv20(idx, inv), c = idx - r * bw;
                            int i = UY0 + r, j = UX0 + c;
                            int u = 0;
                            if ((unsigned)i < (unsigned)H && (unsigned)j < (unsigned)W)
                                u = remap_px(fr, W, H, i, j, (uint32_t)map[(size_t)i * W + j]);
                            S.U[(i - (y0 - HALO_U)) * REG_U + (j - (x0 - HALO_U))] = (uint8_t)u;
                        }
                    }
                    __syncwarp();
                    // ---- 3. horizontal 5-sums of U for rows UY0..UY1, cols BX0..BX1 --------------------
                    {
                        int bw = BX1 - BX0 + 1, n = bw * (UY1 - UY0 + 1), inv = finv20(bw);
                        for (int idx = lane; idx < n; idx += 32) {
                            int r = fdiv20(idx, inv), c = idx - r * bw;
                            int ur = UY0 + r - (y0 - HALO_U), uc = BX0 + c - 2 - (x0 - HALO_U);
                            const uint8_t* u = &S.U[ur * REG_U + uc];
                            S.HS[ur * REG_B + (BX0 + c - (x0 - 2))] = (uint16_t)(u[0] + u[1] + u[2] + u[3] + u[4]);
                        }
                    }
                    __syncwarp();
                }
                // ---- 4. B on the read set: threshold inside the compute box, 0 elsewhere ----------------
                {
                    int bw = RX1 - RX0 + 1, n = bw * (RY1 - RY0 + 1), inv = finv20(bw);
                    for (int idx = lane; idx < n; idx += 32) {
                        int r = fdiv20(idx, inv), c = idx - r * bw;
                        int i = RY0 + r, j = RX0 + c;
                        int b = 0;
                        if (i >= BY0 && i <= BY1 && j >= BX0 && j <= BX1) {
                            int ur = i - 2 - (y0 - HALO_U), bc = j - (x0 - 2);
                            const uint16_t* h = &S.HS[ur * REG_B + bc];
                            int s = h[0] + h[REG_B] + h[2 * REG_B] + h[3 * REG_B] + h[4 * REG_B];
                            int cnt = (min(i + 2, H - 1) - max(i - 2, 0) + 1) * (min(j + 2, W - 1) - max(j - 2, 0) + 1);
                            b = s >= T * cnt;
                        }
                        S.B[(i - (y0 - 2)) * REG_B + (j - (x0 - 2))] = (uint8_t)b;
                    }
                }
                __syncwarp();
                // ---- 5. majority: horizontal 5-sums (clamped columns) into HS, then vertical -------------
                {
                    int bw = MX1 - MX0 + 1, n = bw * (RY1 - RY0 + 1), inv = finv20(bw);
                    for (int idx = lane; idx < n; idx += 32) {
                        int r = fdiv20(idx, inv), c = idx - r * bw;
                        int i = RY0 + r, j = MX0 + c;
                        const uint8_t* b = &S.B[(i - (y0 - 2)) * REG_B - (x0 - 2)];
                        int s = b[max(j - 2, 0)] + b[max(j - 1, 0)] + b[j] + b[min(j + 1, W - 1)] + b[min(j + 2, W - 1)];
                        S.HS[(i - (y0 - 2)) * REG_B + (j - x0)] = (uint16_t)s;
                    }
                }
                __syncwarp();
                {
                    int j = x0 + lane;
                    bool colin = j >= MX0 && j <= MX1;
                    for (int i = MY0; i <= MY1; ++i) {
                        int s = 0;
                        if (colin) {
                            const uint16_t* h = &S.HS[-(y0 - 2) * REG_B + lane];
                            s = h[max(i - 2, 0) * REG_B] + h[max(i - 1, 0) * REG_B] + h[i * REG_B] +
                                h[min(i + 1, H - 1) * REG_B] + h[min(i + 2, H - 1) * REG_B];
                        }
                        unsigned wv = __ballot_sync(0xffffffffu, s >= 13);
                        if (lane == i - y0) myword = wv;
                    }
                }
                __syncwarp();
            }
        }
        // ---- 6. write the tile's 32 words ---------------------------------------------------------------
        if (y0 + lane < H) brow[(size_t)lane * TX] = myword;
        unsigned nz = __ballot_sync(0xffffffffu, myword != 0);
        if (nz) {
            if (lane == 0) {
                int slot = atomicAdd(&n_fg[f], 1);
                if (slot < max_fg) fg_tiles[(size_t)f * max_fg + slot] = (uint32_t)t;
                else atomicOr(&flags[f], MOCAP_FLAG_TILE_OVERFLOW);
            }
            // neighbours that no warp owns must read as background for the border walkers
            if (lane < 8) {
                int k = lane + (lane >= 4);
                int nx = tx + k % 3 - 1, ny = ty + k / 3 - 1;
                bool zero = nx >= 0 && ny >= 0 && nx < TX && ny < TY &&
                            !((active[((size_t)f * TY + ny) * TXW + (nx >> 5)] >> (nx & 31)) & 1);
                if (zero) {
                    uint32_t* nb = bits + ((size_t)f * H + ny * TILE) * TX + nx;
                    for (int r = 0; r < TILE && ny * TILE + r < H; ++r) nb[(size_t)r * TX] = 0;
                }
            }
        }
    }
}

// dense copy-out of the packed binary image (parity / debug output): inactive tiles read as zero
__global__ void materialize_bits_kernel(const uint32_t* __restrict__ bits, const uint32_t* __restrict__ active,
                                        int n_frames, int H, int TX, int TY, int TXW, int W, uint32_t* __restrict__ out)
{
    long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    long long total = (long long)n_frames * H * TX;
    if (idx >= total) return;
    int tx = (int)(idx % TX);
    long long r = idx / TX;
    int y = (int)(r % H), f = (int)(r / H);
    bool act = (active[((size_t)f * TY + (y >> 5)) * TXW + (tx >> 5)] >> (tx & 31)) & 1;
    uint32_t w = act ? bits[idx] : 0u;
    int rem = W - tx * 32;
    if (rem < 32) w &= (1u << rem) - 1u;
    out[idx] = w;
}

// ---------------------------------------------------------------------------------------------------------
// host-side launcher shared by mocap_filter_batch and mocap_detect_batch
// ---------------------------------------------------------------------------------------------------------
int launch_scan(const uint8_t* frames, int n, int /*H*/, int W, int64_t fstride, const TableView& tv, int thresh,
                const FilterWs& ws, cudaStream_t s, StageTimer* timer)
{
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    HotTest ht = make_hot_test(thresh);
    bool vec = (W % 16 == 0) && (fstride % 16 == 0) && (((uintptr_t)frames) % 16 == 0);
    bool vec32 = (W % 32 == 0) && (fstride % 32 == 0) && (((uintptr_t)frames) % 32 == 0);
    stage_begin(timer, 0, s);
    if (vec32) {
        int grid = sms * 4;                      // persistent: exactly the resident CTAs (__launch_bounds__(256, 4)), one wave
        switch (ht.mode) {
            case 0: LAUNCH(scan_hot_vec32_kernel<0>, grid, 256, 0, s, frames, n, fstride, tv, ht.add, ws.cellbox); break;
            case 1: LAUNCH(scan_hot_vec32_kernel<1>, grid, 256, 0, s, frames, n, fstride, tv, ht.add, ws.cellbox); break;
            case 2: LAUNCH(scan_hot_vec32_kernel<2>, grid, 256, 0, s, frames, n, fstride, tv, ht.add, ws.cellbox); break;
            default: LAUNCH(scan_hot_vec32_kernel<3>, grid, 256, 0, s, frames, n, fstride, tv, ht.add, ws.cellbox); break;
        }
    } else if (vec) {
        int grid = sms * 4;
        switch (ht.mode) {
            case 0: LAUNCH(scan_hot_vec_kernel<0>, grid, 256, 0, s, frames, n, fstride, tv, ht.add, ws.cellbox); break;
            case 1: LAUNCH(scan_hot_vec_kernel<1>, grid, 256, 0, s, frames, n, fstride, tv, ht.add, ws.cellbox); break;
            case 2: LAUNCH(scan_hot_vec_kernel<2>, grid, 256, 0, s, frames, n, fstride, tv, ht.add, ws.cellbox); break;
            default: LAUNCH(scan_hot_vec_kernel<3>, grid, 256, 0, s, frames, n, fstride, tv, ht.add, ws.cellbox); break;
        }
    } else {
        LAUNCH(scan_hot_scalar_kernel, sms * 8, 256, 0, s, frames, n, fstride, tv, thresh, ws.cellbox);
    }
    stage_end(timer, 0, s);
    CUDA_TRY(cudaGetLastError());
    return MOCAP_OK;
}

// general path, filter part: active tiles of the frames in need_general (all frames if null) -> packed binary image
int launch_tiles(const uint8_t* frames, int n, int /*H*/, int W, int64_t fstride, const TableView& tv, int thresh,
                 const FilterWs& ws, int max_fg, int* flags, const int* need_general, cudaStream_t s)
{
    const int TX = tv.TX, TY = tv.TY, TXW = cdiv(TX, 32);
    CUDA_TRY(cudaMemsetAsync(ws.counters, 0, 2 * sizeof(int), s));
    CUDA_TRY(cudaMemsetAsync(ws.n_fg, 0, (size_t)n * sizeof(int), s));
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    CUDA_TRY(cudaMemsetAsync(ws.active, 0, (size_t)n * TY * TXW * 4, s));
    LAUNCH(mark_active_kernel, (unsigned)(n < 65535 ? n : 65535), 256, 0, s, ws.cellbox, tv, n, ws.active, TXW, need_general, flags);
    long long n_words = (long long)n * TY * TXW;
    LAUNCH(compact_tiles_kernel, (unsigned)((n_words + 255) / 256), 256, 0, s, ws.active, n_words, TX, TY, TXW, ws.list, ws.counters, need_general);
    LAUNCH(filter_tiles_kernel, sms * 4, FT_WARPS * 32, 0, s, frames, fstride, tv, thresh, ws.list, ws.counters, ws.counters + 1,
                                                          ws.active, TXW, ws.cellbox, ws.bits, ws.fg_tiles, ws.n_fg, max_fg, flags);
    CUDA_TRY(cudaGetLastError());
    return MOCAP_OK;
}

int launch_materialize_bits(const FilterWs& ws, int n, int H, int W, const TableView& tv, uint32_t* out, cudaStream_t s)
{
    long long total = (long long)n * H * tv.TX;
    LAUNCH(materialize_bits_kernel, (unsigned)((total + 255) / 256), 256, 0, s, ws.bits, ws.active, n, H, tv.TX, tv.TY,
           cdiv(tv.TX, 32), W, out);
    CUDA_TRY(cudaGetLastError());
    return MOCAP_OK;
}

// ---------------------------------------------------------------------------------------------------------
// stage kernels for parity tests: the reference's own blur (CudaOperations.py:5-41) and cv.undistort alone
// ---------------------------------------------------------------------------------------------------------
__global__ void blur5_kernel(const uint8_t* __restrict__ in, int n, int H, int W, uint8_t* __restrict__ out)
{
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y, f = blockIdx.z;
    if (x >= W || y >= H) return;
    const uint8_t* fr = in + (size_t)f * H * W;
    int s = 0, c = 0;
    for (int dy = -2; dy <= 2; ++dy)
        for (int dx = -2; dx <= 2; ++dx) {
            int yy = y + dy, xx = x + dx;
            if ((unsigned)yy < (unsigned)H && (unsigned)xx < (unsigned)W) { s += fr[(size_t)yy * W + xx]; ++c; }
        }
    out[(size_t)f * H * W + (size_t)y * W + x] = (uint8_t)(s / c);
}

extern "C" int mocap_blur5_batch(const uint8_t* frames_dev, int n, int H, int W, uint8_t* out_dev, void* stream)
{
    if (!frames_dev || !out_dev || n <= 0 || H <= 0 || W <= 0 || n > 65535) return MOCAP_ERR_INVALID;
    LAUNCH(blur5_kernel, dim3(cdiv(W, 32), cdiv(H, 8), n), dim3(32, 8), 0, (cudaStream_t)stream, frames_dev, n, H, W, out_dev);
    CUDA_TRY(cudaGetLastError());
    return MOCAP_OK;
}

// cv.medianBlur(image, 5) on grey u8 (BORDER_REPLICATE) followed by cv.threshold(., thresh, 255, THRESH_BINARY):
// image_filter_cpu of the reference (lib/ImageOperations.py:15-21; it has no callers there).  One pixel per thread:
// the median is the value whose rank interval covers position 12 of the 25 window values.
__global__ void median5_threshold_kernel(const uint8_t* __restrict__ in, int n, int H, int W, int thresh, uint8_t* __restrict__ out)
{
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y, f = blockIdx.z;
    if (x >= W || y >= H) return;
    const uint8_t* fr = in + (size_t)f * H * W;
    int v[25];
#pragma unroll
    for (int dy = -2; dy <= 2; ++dy)
#pragma unroll
        for (int dx = -2; dx <= 2; ++dx)
            v[(dy + 2) * 5 + dx + 2] = fr[(size_t)min(max(y + dy, 0), H - 1) * W + min(max(x + dx, 0), W - 1)];
    int med = 0;
#pragma unroll
    for (int a = 0; a < 25; ++a) {
        int less = 0, leq = 0;
#pragma unroll
        for (int b = 0; b < 25; ++b) { less += v[b] < v[a]; leq += v[b] <= v[a]; }
        if (less <= 12 && 12 < leq) med = v[a];
    }
    out[(size_t)f * H * W + (size_t)y * W + x] = med > thresh ? 255 : 0;
}

extern "C" int mocap_median5_threshold_batch(const uint8_t* frames_dev, int n, int H, int W, int thresh, uint8_t* out_dev, void* stream)
{
    if (!frames_dev || !out_dev || n <= 0 || H <= 0 || W <= 0 || n > 65535) return MOCAP_ERR_INVALID;
    LAUNCH(median5_threshold_kernel, dim3(cdiv(W, 32), cdiv(H, 8), n), dim3(32, 8), 0, (cudaStream_t)stream, frames_dev, n, H, W, thresh, out_dev);
    CUDA_TRY(cudaGetLastError());
    return MOCAP_OK;
}

// Bayer front step of the realtime loop (RealtimeTracking_FLIR.py:103-104): cvtColor(BAYER_GR2BGR) -> cvtColor(BGR2GRAY),
// fused: raw sensor bytes in, grey bytes out, no BGR intermediate.  Red on (odd row, even column), blue on (even row, odd
// column); OpenCV's bilinear means ((a+b+1)>>1, (a+b+c+d+2)>>2), border rows / columns copy their inner neighbour;
// grey = (9798 R + 19235 G + 3735 B + 16384) >> 15.  One thread per output pixel; neighbours come through L1.
__global__ void bayer_gr2gray_kernel(const uint8_t* __restrict__ in, int n, int H, int W, uint8_t* __restrict__ out)
{
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y, f = blockIdx.z;
    if (x >= W || y >= H) return;
    const uint8_t* fr = in + (size_t)f * H * W;
    int yc = min(max(y, 1), H - 2), xc = min(max(x, 1), W - 2);
    const uint8_t* p = fr + (size_t)yc * W + xc;
    int c = p[0], l = p[-1], r = p[1], u = p[-W], d = p[W];
    int ul = p[-W - 1], ur = p[-W + 1], dl = p[W - 1], dr = p[W + 1];
    int cross = (u + d + l + r + 2) >> 2, diag = (ul + ur + dl + dr + 2) >> 2, hor = (l + r + 1) >> 1, ver = (u + d + 1) >> 1;
    bool odd_row = yc & 1, odd_col = xc & 1;
    int R, G, B;
    if (odd_row && !odd_col) { R = c; G = cross; B = diag; }            // red site
    else if (!odd_row && odd_col) { B = c; G = cross; R = diag; }       // blue site
    else if (odd_row) { G = c; R = hor; B = ver; }                      // green on a red row
    else { G = c; B = hor; R = ver; }                                   // green on a blue row
    out[(size_t)f * H * W + (size_t)y * W + x] = (uint8_t)((R * 9798 + G * 19235 + B * 3735 + 16384) >> 15);
}

// The same conversion at streaming speed (rows that are a multiple of 4 bytes, 4-byte aligned buffers): a warp walks a
// strip of BAYER_ROWS rows top to bottom, a lane owns NW consecutive 32-bit words of a row (4 NW pixels).  Every input byte is
// loaded once, two rows ahead of its use; the words left and right of a lane's span come from the adjacent lanes by shuffle
// (lanes 0 / 31 fetch theirs with the row).  A row is kept as four registers per word, each holding two pixels as 16-bit
// lanes: the even pixels (x, x+2), the odd pixels (x+1, x+3), and the pairs (x-1, x+1) / (x+2, x+4) -- the left neighbours of
// the even and the right neighbours of the odd pixels; the other two neighbour pairs ARE the odd / even pixels.  With the word
// on an even column, the even pixels of a row are all the same kind of site (red or green) and the odd pixels the other, so
// the bilinear means run on both pixels of a register at once (sums <= 1022 fit the 16-bit lanes; the shifted sums are
// consumed byte-wise, so the bits that cross a lane need no mask).  Grey: the weights doubled (19596 R + 38470 G + 7470 B +
// 32768 <= 2^24 - 32768) put the result into byte 2 of the sum, i.e. three IDP.2A per pixel (FMA pipe) and no shift; three PRMT
// assemble the four bytes of a word, the last one with a per-lane selector that also copies column 1 to column 0 and column
// W-2 to column W-1.  Rows 0 and H-1 (copies of rows 1 and H-2) are stored by the warps that produce rows 1 and H-2.
#ifndef BAYER_MIN_CTAS
#define BAYER_MIN_CTAS 1                                      // (9 / 10 cap the registers at 56 / 48: 0.46 / 0.45 ms against 0.436 per 256 frames)
#endif
#ifndef BAYER_ROWS
#define BAYER_ROWS 64
#endif
#ifndef BAYER_DEPTH
#define BAYER_DEPTH 3                                          // input rows in flight per thread (a divisor of 6); 2: 0.457, 3: 0.436, 6: 0.495 ms per 256 frames of 2048x2048
#endif
struct BayerRow { uint32_t wE, wO, lE, rO; };                  // pixels (x, x+2), (x+1, x+3), (x-1, x+1), (x+2, x+4) of a word at x
template <int NW> struct BayerRows { BayerRow w[NW]; };
template <int NW> struct BayerRaw { uint32_t w[NW], prev, next; };       // a thread's words of a row + the words left / right of them

// eL / eR: byte offsets of the neighbour words (-4 / 4 NW; 0 / 4 NW - 4 for the thread at a row end while the frame's first /
// last row is loaded, where the neighbour word would lie outside the buffer: its bytes only reach the copied columns)
template <int NW>
__device__ __forceinline__ void bayer_load(const uint8_t* __restrict__ p, int eL, int eR, BayerRaw<NW>& r)
{
    if (NW == 2) { uint2 v = *(const uint2*)p; r.w[0] = v.x; r.w[NW - 1] = v.y; }
    else r.w[0] = *(const uint32_t*)p;
    r.prev = *(const uint32_t*)(p + eL);
    r.next = *(const uint32_t*)(p + eR);
}

template <int NW>
__device__ __forceinline__ BayerRows<NW> bayer_split(const BayerRaw<NW>& raw)
{
    BayerRows<NW> r;
#pragma unroll
    for (int k = 0; k < NW; ++k) {
        const uint32_t w = raw.w[k];
        r.w[k].wE = __byte_perm(w, 0, 0x4240);
        r.w[k].wO = __byte_perm(w, 0, 0x4341);
        r.w[k].lE = __byte_perm(k == 0 ? raw.prev : raw.w[k > 0 ? k - 1 : 0], r.w[k].wO, 0x5453);
        r.w[k].rO = __byte_perm(r.w[k].wE, k == NW - 1 ? raw.next : raw.w[k < NW - 1 ? k + 1 : k], 0x1412);
    }
    return r;
}

// grey bytes of the two pixels of a register: R / G / B as 16-bit lanes whose bytes 0 and 2 hold the values (bytes 1 and 3 may
// carry stray bits: their weight is zero) -> sums with the grey byte in bits 16..23.  One IDP.2A per channel and pixel: the
// FMA pipe has room, the ALU pipe (PRMT, shifts, adds) is the one that fills, so nothing is packed first.
__device__ __forceinline__ void bayer_grey2(uint32_t Rp, uint32_t Gp, uint32_t Bp, uint32_t& s0, uint32_t& s1)
{
    const uint32_t WR = 19596u, WG = 38470u, WB = 7470u;               // 2 x (9798, 19235, 3735); high halves (bytes 1 / 3) zero
    s0 = __dp2a_lo(WR, Rp, __dp2a_lo(WG, Gp, __dp2a_lo(WB, Bp, 32768u)));
    s1 = __dp2a_hi(WR, Rp, __dp2a_hi(WG, Gp, __dp2a_hi(WB, Bp, 32768u)));
}

// grey word (4 pixels) of an output row from the rows above / at / below it; `odd`: row parity (red row); `sel`: byte
// selector of the last PRMT (0x5410, or the edge copies)
__device__ __forceinline__ uint32_t bayer_row_grey(const BayerRow& u, const BayerRow& c, const BayerRow& d, bool odd, uint32_t sel)
{
    const uint32_t C1 = 0x00010001u, C2 = 0x00020002u;
    uint32_t e0, e1, o0, o1;                                           // sums of the even / odd pixels of the word
    if (odd) {
        // red row: even pixels are red sites (G = cross, B = diagonals), odd pixels green (R = horizontal, B = vertical)
        const uint32_t vO = u.wO + d.wO + C1;
        const uint32_t cross = (u.wE + d.wE + C2 + c.lE + c.wO) >> 2, diag = (u.lE + d.lE + C1 + vO) >> 2;
        const uint32_t hor = (c.wE + c.rO + C1) >> 1, ver = vO >> 1;
        bayer_grey2(c.wE, cross, diag, e0, e1);
        bayer_grey2(hor, c.wO, ver, o0, o1);
    } else {
        // blue row: even pixels green (B = horizontal, R = vertical), odd pixels blue sites (G = cross, R = diagonals)
        const uint32_t vE = u.wE + d.wE + C1;
        const uint32_t hor = (c.lE + c.wO + C1) >> 1, ver = vE >> 1;
        const uint32_t cross = (u.wO + d.wO + C2 + c.wE + c.rO) >> 2, diag = (u.rO + d.rO + C1 + vE) >> 2;
        bayer_grey2(ver, c.wE, hor, e0, e1);
        bayer_grey2(diag, cross, c.wO, o0, o1);
    }
    return __byte_perm(__byte_perm(e0, o0, 0x0062), __byte_perm(e1, o1, 0x0062), sel);
}

// interior rows 1 .. H-2 (+ rows 0 and H-1, their copies); NW words (4 NW pixels) per thread and row; the threads of a block
// lie side by side on one strip of rows (grid: x = spans of 128 threads, y = strips, z = frames)
// SCAN: the kernel also does the streaming scan of the detection on the grey bytes it holds -- per 32x32 cell of the grey frame the
// masks of its hot columns and rows (pixel > thresh, the test of scan_hot_*_kernel) are OR-ed into cellmask [n][TY][TX][2];
// pack_cellmask_kernel turns them into the cell boxes.  A row without a byte >= 128 costs one LOP3 and a branch (thresh >= 128: the
// detection's threshold is 216); rows with hot pixels are rare (the markers) and issue two RED.OR per thread.
struct BayerScan { uint32_t* cellmask; uint32_t add; int mode; int TX, TY; };
template <int NW, bool SCAN>
__global__ void __launch_bounds__(128, BAYER_MIN_CTAS) bayer_gr2gray_rows_kernel(const uint8_t* __restrict__ in, int H, int W, uint8_t* __restrict__ out, BayerScan sc)
{
    const int x0 = (blockIdx.x * 128 + threadIdx.x) * 4 * NW;
    const int ya = max((int)blockIdx.y * BAYER_ROWS, 1), yb = min(((int)blockIdx.y + 1) * BAYER_ROWS, H - 1);   // interior output rows [ya, yb)
    if (x0 >= W || ya >= yb) return;
    const uint8_t* p = in + (size_t)blockIdx.z * H * W + (size_t)(ya - 1) * W + x0;           // walks down the input rows
    uint8_t* q = out + (size_t)blockIdx.z * H * W + (size_t)ya * W + x0;                      // walks down the output rows
    // column 0 copies column 1, column W-1 copies column W-2: selectors of the first / last word's last PRMT
    const uint32_t sel_first = (x0 == 0 ? 0x5411u : 0x5410u) & (NW == 1 && x0 + 4 == W ? 0x4fffu : 0xffffu);
    const uint32_t sel_last = NW == 1 ? sel_first : (x0 + 4 * NW == W ? 0x4410u : 0x5410u);
    const int eL = x0 == 0 ? 0 : -4, eR = x0 + 4 * NW == W ? 4 * NW - 4 : 4 * NW;
    BayerRows<NW> r[3];
    BayerRaw<NW> fl[BAYER_DEPTH];                                      // the next BAYER_DEPTH input rows are always in flight; fl[0] the oldest
    int yl = ya - 1;                                                   // the last row requested
    int ysc = ya;                                                      // (SCAN) the next row to be stored
    auto request = [&](BayerRaw<NW>& t) { if (yl + 1 < H) { ++yl; p += W; } bayer_load<NW>(p, eL, eR, t); };
    auto request_fast = [&](BayerRaw<NW>& t) { ++yl; p += W; bayer_load<NW>(p, -4, 4 * NW, t); };     // a row of 1 .. H-2
    auto next_row = [&]() -> BayerRows<NW> {                           // outside the unrolled loop: consume fl[0], request, rotate
        BayerRows<NW> t = bayer_split<NW>(fl[0]);
        request(fl[0]);
        BayerRaw<NW> o = fl[0];
#pragma unroll
        for (int k = 0; k + 1 < BAYER_DEPTH; ++k) fl[k] = fl[k + 1];
        fl[BAYER_DEPTH - 1] = o;
        return t;
    };
    bayer_load<NW>(p, eL, eR, fl[0]);
#pragma unroll
    for (int k = 1; k < BAYER_DEPTH; ++k) request(fl[k]);
    r[0] = next_row();
    r[1] = next_row();
    auto store = [&](uint8_t* t, const uint32_t g[NW]) {
        if (NW == 2) *(uint2*)t = make_uint2(g[0], g[NW - 1]);
        else *(uint32_t*)t = g[0];
    };
    // `top` / `bottom`: the row is row 1 / row H-2 and is stored to row 0 / row H-1 as well
    auto emit = [&](const BayerRows<NW>& u, const BayerRows<NW>& c, const BayerRows<NW>& d, bool odd, bool top, bool bottom) {
        uint32_t g[NW];
#pragma unroll
        for (int k = 0; k < NW; ++k)
            g[k] = bayer_row_grey(u.w[k], c.w[k], d.w[k], odd, k == 0 ? sel_first : k == NW - 1 ? sel_last : 0x5410u);
        store(q, g);
        if (top) store(q - W, g);
        if (bottom) store(q + W, g);
        q += W;
        if (SCAN) {
            uint32_t any = g[0];
#pragma unroll
            for (int k = 1; k < NW; ++k) any |= g[k];
            if (((any & 0x80808080u) != 0 && sc.mode != 2) || (sc.mode & 1)) {          // (modes 1 / 3: thresh < 128, every row is tested)
                uint32_t cm = 0;
#pragma unroll
                for (int k = 0; k < NW; ++k) {
                    const uint32_t t = (g[k] & 0x7f7f7f7fu) + sc.add;
                    const uint32_t h = sc.mode == 0 ? (g[k] & t) : sc.mode == 1 ? (g[k] | t) : 0x80808080u;
                    cm |= hot_nibble(h) << (4 * k);
                }
                if (cm) {
                    const int ys = ysc;                                    // the row just stored
                    auto mark = [&](int row) {
                        uint32_t* m = sc.cellmask + 2 * (((size_t)blockIdx.z * sc.TY + (row >> 5)) * sc.TX + (x0 >> 5));
                        atomicOr(m, cm << (x0 & 31));
                        atomicOr(m + 1, 1u << (row & 31));
                    };
                    mark(ys);
                    if (top) mark(ys - 1);
                    if (bottom) mark(ys + 1);
                }
            }
            ++ysc;
        }
    };
    int y = ya;
    if (y & 1) {                                                       // first strip (ya = 1): start the unrolled loop on an even row
        r[2] = next_row();
        emit(r[0], r[1], r[2], true, true, y == H - 2);
        r[0] = r[1]; r[1] = r[2];
        ++y;
    }
    // six rows per pass: the three row registers and the rows in flight rotate back to where they started and the row parity
    // is a constant; the pass requests rows up to y + 6 + BAYER_DEPTH <= H - 2 without a test (neighbour words at fixed
    // offsets), and at least one row is left to the loop below (the one that may be row H-2)
    for (const int ye = min(yb - 7, H - 8 - BAYER_DEPTH); y <= ye; y += 6) {
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            r[(k + 2) % 3] = bayer_split<NW>(fl[k % BAYER_DEPTH]);
            request_fast(fl[k % BAYER_DEPTH]);
            emit(r[k % 3], r[(k + 1) % 3], r[(k + 2) % 3], (k & 1) != 0, false, false);
        }
    }
    for (; y < yb; ++y) {
        r[2] = next_row();
        emit(r[0], r[1], r[2], (y & 1) != 0, false, y == H - 2);
        r[0] = r[1]; r[1] = r[2];
    }
}

__global__ void pack_cellmask_kernel(const uint32_t* __restrict__ cellmask, long long cells, uint32_t* __restrict__ cellbox)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < cells) cellbox[i] = pack_cellbox(cellmask[2 * i], cellmask[2 * i + 1]);
}

// grey frames (+ with cellbox_out: the hot cell boxes of the grey frames for `thresh`, what the streaming scan of the detection
// would compute from them; scan_ws >= n * ceil(H/32) * ceil(W/32) * 8 bytes)
static int bayer_launch(const uint8_t* raw_dev, int n, int H, int W, uint8_t* out_dev, int thresh, uint32_t* cellbox_out, void* scan_ws,
                        size_t scan_ws_bytes, cudaStream_t st)
{
    if (!raw_dev || !out_dev || n <= 0 || H < 3 || W < 3 || n > 65535 || (long long)H * W >= (1ll << 31)) return MOCAP_ERR_INVALID;
    const uintptr_t al = (uintptr_t)raw_dev | (uintptr_t)out_dev | (uintptr_t)W;
    BayerScan sc = {nullptr, 0u, 2, (W + 31) / 32, (H + 31) / 32};
    const long long cells = (long long)n * sc.TX * sc.TY;
    const bool scan = cellbox_out != nullptr;
    if (scan) {
        if (!scan_ws || scan_ws_bytes < (size_t)cells * 8) return MOCAP_ERR_WORKSPACE;
        HotTest ht = make_hot_test(thresh);
        sc.cellmask = (uint32_t*)scan_ws; sc.add = ht.add; sc.mode = ht.mode;
    }
    if (al % 4 == 0) {
        const int ny = cdiv(H, BAYER_ROWS);
        if (scan) CUDA_TRY(cudaMemsetAsync(scan_ws, 0, (size_t)cells * 8, st));
        // (four words per thread -- 128-bit loads, 88-96 registers -- measured slower: 0.44-0.47 ms against 0.436 per 256 frames)
        if (al % 8 == 0) {
            if (scan) LAUNCH((bayer_gr2gray_rows_kernel<2, true>), dim3(cdiv(W, 1024), ny, n), 128, 0, st, raw_dev, H, W, out_dev, sc);
            else LAUNCH((bayer_gr2gray_rows_kernel<2, false>), dim3(cdiv(W, 1024), ny, n), 128, 0, st, raw_dev, H, W, out_dev, sc);
        } else {
            if (scan) LAUNCH((bayer_gr2gray_rows_kernel<1, true>), dim3(cdiv(W, 512), ny, n), 128, 0, st, raw_dev, H, W, out_dev, sc);
            else LAUNCH((bayer_gr2gray_rows_kernel<1, false>), dim3(cdiv(W, 512), ny, n), 128, 0, st, raw_dev, H, W, out_dev, sc);
        }
        if (scan) LAUNCH(pack_cellmask_kernel, (unsigned)((cells + 255) / 256), 256, 0, st, (const uint32_t*)scan_ws, cells, cellbox_out);
        CUDA_TRY(cudaGetLastError());
        return MOCAP_OK;
    }
    LAUNCH(bayer_gr2gray_kernel, dim3(cdiv(W, 64), cdiv(H, 4), n), dim3(64, 4), 0, st, raw_dev, n, H, W, out_dev);
    CUDA_TRY(cudaGetLastError());
    if (scan) {                                                            // rows that are not a multiple of 4 bytes: the generic scan on the grey frames
        TableView tv = {};
        tv.H = H; tv.W = W; tv.TX = sc.TX; tv.TY = sc.TY;                  // (the scalar scan reads the frame geometry only)
        LAUNCH(scan_hot_scalar_kernel, 148 * 8, 256, 0, st, (const uint8_t*)out_dev, n, (int64_t)H * W, tv, thresh, cellbox_out);
        CUDA_TRY(cudaGetLastError());
    }
    return MOCAP_OK;
}

extern "C" int mocap_bayer_gr2gray_batch(const uint8_t* raw_dev, int n, int H, int W, uint8_t* out_dev, void* stream)
{
    return bayer_launch(raw_dev, n, H, W, out_dev, 0, nullptr, nullptr, 0, (cudaStream_t)stream);
}

extern "C" int mocap_bayer_gr2gray_scan_batch(const uint8_t* raw_dev, int n, int H, int W, uint8_t* out_dev, int thresh,
                                              uint32_t* cellbox_out, void* workspace, size_t workspace_bytes, void* stream)
{
    if (!cellbox_out) return MOCAP_ERR_INVALID;
    return bayer_launch(raw_dev, n, H, W, out_dev, thresh, cellbox_out, workspace, workspace_bytes, (cudaStream_t)stream);
}

__global__ void undistort_kernel(const uint8_t* __restrict__ in, int n, int H, int W, const int32_t* __restrict__ map,
                                 uint8_t* __restrict__ out)
{
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y, f = blockIdx.z;
    if (x >= W || y >= H) return;
    out[(size_t)f * H * W + (size_t)y * W + x] =
        (uint8_t)remap_px(in + (size_t)f * H * W, W, H, y, x, (uint32_t)map[(size_t)y * W + x]);
}

extern "C" int mocap_undistort_batch(const uint8_t* frames_dev, int n, int H, int W, const void* table_dev,
                                     uint8_t* out_dev, void* stream)
{
    if (!frames_dev || !out_dev || !table_dev || n <= 0 || H <= 0 || W <= 0 || n > 65535) return MOCAP_ERR_INVALID;
    TableView tv; table_view(table_dev, H, W, &tv);
    LAUNCH(undistort_kernel, dim3(cdiv(W, 32), cdiv(H, 8), n), dim3(32, 8), 0, (cudaStream_t)stream, frames_dev, n, H, W, tv.map, out_dev);
    CUDA_TRY(cudaGetLastError());
    return MOCAP_OK;
}
