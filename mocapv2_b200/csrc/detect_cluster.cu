// Cluster path of _find_dot (the product path): after the streaming scan, every group of hot 32x32 source cells is
// handled as ONE unit entirely in shared memory -- remap + 5x5 floor-mean threshold + 5x5 majority on the group's
// output box, border starts from the rows' bit masks, Suzuki-Abe trace, Green sums -- and appends one record per outer
// border to the frame's list.  A small per-frame kernel then applies the reference's filter / centroid / output order
// (lib/ImageOperations.py:38-65).  No per-frame serial stage and no round trip of the binary image through HBM.
//
// Exactness: (1) a filtered pixel can only be set within reach of a source pixel > thresh, so every foreground pixel lies
// inside the output box of some hot cell; (2) a cluster is a connected component of the "boxes touch" graph over the hot
// cells, so two 8-adjacent foreground pixels always lie in boxes of the same cluster: a blob is covered by the boxes of
// exactly one cluster and no foreground pixel of another cluster lies inside them.  A cluster therefore filters the
// bounding box of its (tighter, +-2) boxes and reports exactly the borders whose start pixel lies inside one of its own +-4
// boxes (the bounding box may show parts of foreign blobs; they are never owned).  What a unit cannot decide locally (a hole
// border -> contour tree, a group larger than the largest size class, capacity overflows) flags the FRAME for the
// general per-frame path (detect_filter.cu + detect_blobs.cu), which recomputes it from the source frame.
#include "common.cuh"
#include "remap.cuh"
#include "walk.cuh"
#include "tma.cuh"

#define CL_THREADS 128
#ifndef BORDERS_MIN_CTAS
#define BORDERS_MIN_CTAS 1                                        // (8 caps borders_finalize_kernel at 64 registers: build-time A/B)
#endif
#ifndef PF_WIN_L2_PROMO
#define PF_WIN_L2_PROMO 64      // bytes a window fetch is widened to in L2 (rows are 96 bytes; 64: 0.99 GB of DRAM reads per 1024 frames, 128 or none: 1.30 GB)
#endif
#ifndef PF_MAP_EVICT
#define PF_MAP_EVICT evict_last // L2 priority of the fast-map reads (build-time A/B: evict_normal, see tools/lens_probe.py)
#endif
#ifndef BF_THREADS
#define BF_THREADS 128          // threads of a border CTA (one frame): with fewer threads a lane follows several borders one after the other
#endif
#define HOT_MAX 1024            // hot cells per frame on the cluster path
#define CELLS_MAX 8192          // TX*TY limit of the dense cell -> slot map held in shared memory
#define ROOTS_MAX 512
#define PIECE 64                // a cluster box is filtered in pieces of at most PIECE x PIECE output pixels
                                // staged source window of a piece: up to WIN_W (96, common.cuh) x 78 bytes (sized so that 8 CTAs fit one SM)
#define WIN_H 78
#define WIN_H_LOW 56            // second TMA box height: most pieces need no more window rows
#define CAND_PER_FRAME 512      // border-start candidates per frame on the cluster path

// counters[] slots
#define CN_CLUSTERS 0
#define CN_PIECES 1
#define CN_PIECE_CUR 2
#define CN_CANDS 3
#define CN_ROWS 4               // words of bit-row storage handed out

struct ClusterWs {
    int* need_general;          // [n] != 0: frame takes the general path (value = why)
    int* counters;              // [16]
    int* clusters;              // [cl_cap][8]: frame, x0 | y0 << 16, x1 | y1 << 16 (box, inclusive), rows word offset, words per row,
                                //              member offset | count << 16, 0, 0
    int* pieces;                // [pc_cap][8]: piece descriptors (make_piece_desc)
    int cl_cap, pc_cap;
    short* memb;                // [n][HOT_MAX][4] output boxes of the hot cells, grouped by cluster
    uint32_t* rows_out;         // filtered bit rows of every cluster box
    unsigned rows_cap;          // words
    int* cand_list;             // [n][CAND_PER_FRAME][2]: cluster, lx | ly << 16 | type << 31
    int* cand_count;            // [n]
    int* frame_clusters;        // [n][2]: first cluster id of the frame, number of clusters (contiguous ids)
    int n_frames;
    int* rec_count;             // [n]
    int* rec_start;             // [n][max_contours] start pixel index y * W + x of an outer border
    long long* rec_a;           // [n][max_contours][3] a00 a10 a01
    double* rec_per;            // [n][max_contours]
    int* rec_info;              // [n][max_contours][4]: is_hole, start pixel of the parent outer border (holes), bbox x0 | y0 << 16, x1 | y1 << 16
};

__device__ __forceinline__ int suf_find(int* parent, int x)
{
    int p = parent[x];
    while (p != x) {
        int g = parent[p];
        if (g != p) parent[x] = g;
        x = p; p = g;
    }
    return x;
}
__device__ __forceinline__ void suf_union(int* parent, int a, int b)
{
    for (;;) {
        a = suf_find(parent, a);
        b = suf_find(parent, b);
        if (a == b) return;
        if (a < b) { int t = a; a = b; b = t; }
        int old = atomicMin(&parent[a], b);
        if (old == a) return;
        a = old;
    }
}

__device__ __forceinline__ int cdiv_dev(int a, int b) { return (a + b - 1) / b; }

// u16 slots of form_clusters_kernel's cell -> hot-slot map; at least two int arrays of HOT_MAX (reused once the map is dead)
__host__ __device__ __forceinline__ int form_idx_slots(int cells) { int a = (cells + 7) & ~7; return a > 4 * HOT_MAX ? a : 4 * HOT_MAX; }

__device__ __forceinline__ bool boxes_touch(const int* a, const int* b)
{
    return a[0] <= b[2] + 1 && b[0] <= a[2] + 1 && a[1] <= b[3] + 1 && b[1] <= a[3] + 1;
}

// Descriptor of one filter piece (<= 64x64 output pixels of a cluster box), everything piece_filter_kernel needs in 32 bytes:
//   [0] frame            [1] px0 | py0 << 16 (piece origin)
//   [2] mw | mh << 8 | hl << 16 | hr << 18 | ht << 20 | hb << 22 | packed << 24 | window fits << 25 | fast map usable << 26
//   [3] word offset of the piece's first bit-row word      [4] words per row | window rows << 16 | 16-byte vectors per row << 24
//   [5] window origin x (s16) | y << 16      [6] lens of the frame (its table lies [6] * lens_words words beyond lens 0's)
// hl, hr, ht, hb (0 or 2): how far the thresholded-mean box extends beyond the piece; it stops at the cluster box.
// packed: no frame border within reach of the piece, the tight boxes apply; else the +-4 box with clamped coordinates.
// window = the source pixels the undistortion of the piece's U box can touch (displacement bounds of the tiles it overlaps).
__device__ __forceinline__ void make_piece_desc(const TableView& tv, int f, int lens, int cx0, int cy0, int cx1, int cy1, int bx, int by,
                                                unsigned cluster_rows, int wpr, int* __restrict__ d)
{
    const int W = tv.W, H = tv.H;
    const int px0 = cx0 + bx * PIECE, py0 = cy0 + by * PIECE;
    const int px1 = min(px0 + PIECE - 1, cx1), py1 = min(py0 + PIECE - 1, cy1);
    const int mw = px1 - px0 + 1, mh = py1 - py0 + 1;
    const int hl = px0 - max(px0 - 2, cx0), hr = min(px1 + 2, cx1) - px1, ht = py0 - max(py0 - 2, cy0), hb = min(py1 + 2, cy1) - py1;
    const bool packed = px0 - hl >= 2 && py0 - ht >= 2 && px1 + hr + 2 < W && py1 + hb + 2 < H;
    const int ux0 = packed ? px0 - hl - 2 : px0 - 4, uy0 = packed ? py0 - ht - 2 : py0 - 4;
    int ux1 = packed ? px1 + hr + 2 : px1 + 4;
    const int uy1 = packed ? py1 + hb + 2 : py1 + 4;
    // the fast remap of the piece filter works on quads of four pixels aligned to frame columns that are multiples of four: its box is
    // padded to such columns on both sides, and the window and the fast-map test below cover the padding (computed, never used)
    const int ux0p = ux0 & ~3, ux1p = ((ux1 + 4) & ~3) - 1;                // quads are aligned to frame columns that are multiples of 4
    const bool padded = packed && ux1p < W;
    const int ux0w = padded ? ux0p : ux0;                                  // the box the window and the fast-map test have to cover
    if (padded) ux1 = ux1p;
    const int tx0 = max(ux0w >> 5, 0), tx1 = min(ux1 >> 5, tv.TX - 1), ty0 = max(uy0 >> 5, 0), ty1 = min(uy1 >> 5, tv.TY - 1);
    int dx0 = 0x7fffffff, dx1 = -0x7fffffff, dy0 = 0x7fffffff, dy1 = -0x7fffffff, no_fast = 0;
    for (int ty = ty0; ty <= ty1; ++ty) {                                  // the U box (<= 72 wide) spans at most 4 tiles per row:
        int4 t[4]; int tf[4];                                              // four loads in flight, surplus ones repeat the last tile
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            t[q] = *(const int4*)(tv.tile + 8 * (ty * tv.TX + min(tx0 + q, tx1)) + 4);
            tf[q] = tv.tflag[ty * tv.TX + min(tx0 + q, tx1)];
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            if (t[q].x <= t[q].y) { dx0 = min(dx0, t[q].x); dx1 = max(dx1, t[q].y); dy0 = min(dy0, t[q].z); dy1 = max(dy1, t[q].w); }
            no_fast |= tf[q];
        }
    }
    int wx0 = 0, wy0 = 0, wh = 0, nvec = 0;
    bool fits = false;
    if (dx0 <= dx1 && tx1 - tx0 <= 3) {
        wx0 = (ux0w + dx0) & ~15; wy0 = uy0 + dy0;
        const int wx1 = ux1 + dx1 + 1, wy1 = uy1 + dy1 + 1;
        fits = wx1 - wx0 + 1 <= WIN_W && wy1 - wy0 + 1 <= WIN_H && wx0 >= -32768 && wy0 >= -32768;
        if (fits) { wh = wy1 - wy0 + 1; nvec = (wx1 - wx0 + 16) >> 4; }
    }
    if (!fits) { wx0 = 0; wy0 = 0; }
    int4 lo, hi;
    lo.x = f;
    lo.y = px0 | (py0 << 16);
    lo.z = mw | (mh << 8) | (hl << 16) | (hr << 18) | (ht << 20) | (hb << 22) | ((int)packed << 24) | ((int)fits << 25) |
           ((int)(padded && fits && !no_fast) << 26);
    lo.w = (int)(cluster_rows + (unsigned)(py0 - cy0) * (unsigned)wpr + (unsigned)(bx * (PIECE / 32)));
    hi.x = wpr | (wh << 16) | (nvec << 24);
    hi.y = (wx0 & 0xffff) | (wy0 << 16);
    hi.z = lens; hi.w = 0;
    *(int4*)d = lo;
    *(int4*)(d + 4) = hi;
}

// ---------------------------------------------------------------------------------------------------------
// per frame: hot cells -> clusters (connected components of "output boxes touch") -> cluster table + filter pieces
// ---------------------------------------------------------------------------------------------------------
// The frame's lens is resolved here, once: the cluster entries and piece descriptors carry it to the later stages.
__global__ void __launch_bounds__(CL_THREADS) form_clusters_kernel(const uint32_t* __restrict__ cellbox, TableView tv_set, ClusterWs cw,
                                                                   int32_t* __restrict__ out_flags)
{
    DYN_SHARED(smraw);
    const int f = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    const int TX = tv_set.TX, TY = tv_set.TY, cells = TX * TY, W = tv_set.W, H = tv_set.H;
    if (cw.need_general[f]) return;
    const int lens = frame_lens_of(tv_set, f);
    if (lens < 0) { if (tid == 0) out_flags[f] |= MOCAP_FLAG_LENS_INDEX; return; }      // no clusters: the border stage writes count 0
    const TableView tv = lens_table(tv_set, lens);
    // carve: idx_of[cells] u16 | hot_cell[HOT_MAX] u16 | parent[HOT_MAX] int | box[HOT_MAX][4] short | cbox[HOT_MAX][4] int | roots[ROOTS_MAX] u16
    uint16_t* idx_of = (uint16_t*)smraw;                // dead after the neighbour pass: its memory then holds fill[] and ymax[]
    uint16_t* hot_cell = idx_of + form_idx_slots(cells);
    int* parent = (int*)(hot_cell + HOT_MAX);
    int* cbox = parent + HOT_MAX;
    short* box = (short*)(cbox + 4 * HOT_MAX);
    uint16_t* roots = (uint16_t*)(box + 4 * HOT_MAX);
    int* r_words = (int*)(roots + ROOTS_MAX);           // per root: bit-row words, pieces, y1 of the box
    int* r_pcs = r_words + ROOTS_MAX;
    int* r_y1 = r_pcs + ROOTS_MAX;
    short* tight = (short*)(r_y1 + ROOTS_MAX);          // [HOT_MAX][4] the +-2 boxes (filter region), see below
    __shared__ int s_nhot, s_nroots, s_bad;
    if (tid == 0) { s_nhot = 0; s_bad = 0; }
    for (int c = tid; c < cells; c += nt) idx_of[c] = 0xffff;
    __syncthreads();
    const uint32_t* cb = cellbox + (size_t)f * cells;
    for (int c = tid; c < cells; c += nt) {
        if (cb[c] != CELL_EMPTY) {
            int slot = atomicAdd(&s_nhot, 1);
            if (slot < HOT_MAX) { hot_cell[slot] = (uint16_t)c; idx_of[c] = (uint16_t)slot; }
        }
    }
    __syncthreads();
    const int n_hot = s_nhot;
    if (n_hot > HOT_MAX) { if (tid == 0) cw.need_general[f] = 2; return; }
    if (n_hot == 0) return;
    // output box of every hot cell: pixels whose filtered value can depend on the cell's hot pixels
    for (int h = tid; h < n_hot; h += nt) {
        int c = hot_cell[h], cy = c / TX, cx = c - cy * TX;
        uint32_t b = cb[c];
        const int32_t* inv = tv.cellinv + 4 * c;
        int hx0 = cx * 32 + (int)(b & 0xff), hx1 = cx * 32 + (int)((b >> 8) & 0xff);
        int hy0 = cy * 32 + (int)((b >> 16) & 0xff), hy1 = cy * 32 + (int)(b >> 24);
        // Undistorted pixels > thresh lie in [hx0 - 1 - dmax, hx1 - dmin] (a hot tap is needed); the thresholded mean can be
        // set at most 2 beyond them and the majority at most 2 beyond that: every foreground pixel lies inside the +-4 box of
        // some hot cell.  These boxes define the clusters and the ownership of a border.
        int ux0 = hx0 - 1 - inv[1], ux1 = hx1 - inv[0], uy0 = hy0 - 1 - inv[3], uy1 = hy1 - inv[2];
        int x0 = ux0 - 4, x1 = ux1 + 4, y0 = uy0 - 4, y1 = uy1 + 4;
        // The region a cluster has to FILTER is tighter: all hot pixels within 4 of a foreground pixel belong to its cluster
        // (their +-4 boxes share that pixel), and 3 beyond the cluster's hot pixels only two columns (rows) of the 5x5 majority
        // window can hold set means, 10 < 13.  So the bounding box of the +-2 boxes holds all of the cluster's foreground.
        int tx0 = ux0 - 2, tx1 = ux1 + 2, ty0 = uy0 - 2, ty1 = uy1 + 2;
        if (inv[0] > inv[1]) { x0 = 1; x1 = 0; }                 // no output pixel samples this cell
        // Clusters are grown over 8-neighbour cells only: boxes of cells two apart must not be able to touch.  That holds while
        // the displacement varies by at most 8 px inside a cell (margin <= 13 per side, hot pixels >= 33 apart); a lens that
        // bends more than that goes to the general path.
        else if (inv[1] - inv[0] > 8 || inv[3] - inv[2] > 8) s_bad = 1;
        x0 = max(x0, 0); y0 = max(y0, 0); x1 = min(x1, W - 1); y1 = min(y1, H - 1);
        tx0 = max(tx0, 0); ty0 = max(ty0, 0); tx1 = min(tx1, W - 1); ty1 = min(ty1, H - 1);
        if (x0 > x1 || y0 > y1 || tx0 > tx1 || ty0 > ty1) { x0 = 1; x1 = 0; y0 = 1; y1 = 0; }
        box[4 * h] = (short)x0; box[4 * h + 1] = (short)y0; box[4 * h + 2] = (short)x1; box[4 * h + 3] = (short)y1;
        tight[4 * h] = (short)tx0; tight[4 * h + 1] = (short)ty0; tight[4 * h + 2] = (short)tx1; tight[4 * h + 3] = (short)ty1;
        parent[h] = h;
    }
    __syncthreads();
    if (s_bad) { if (tid == 0) cw.need_general[f] = 10; return; }
    // first grouping: hot 8-neighbour cells whose boxes touch
    for (int h = tid; h < n_hot; h += nt) {
        if (box[4 * h] > box[4 * h + 2]) continue;
        int c = hot_cell[h], cy = c / TX, cx = c - cy * TX;
        int a[4] = {box[4 * h], box[4 * h + 1], box[4 * h + 2], box[4 * h + 3]};
        const int ndx[4] = {-1, -1, 0, 1}, ndy[4] = {0, -1, -1, -1};
        for (int q = 0; q < 4; ++q) {
            int nx = cx + ndx[q], ny = cy + ndy[q];
            if (nx < 0 || ny < 0 || nx >= TX) continue;
            int k = idx_of[ny * TX + nx];
            if (k == 0xffff || box[4 * k] > box[4 * k + 2]) continue;
            int bb[4] = {box[4 * k], box[4 * k + 1], box[4 * k + 2], box[4 * k + 3]};
            if (boxes_touch(a, bb)) suf_union(parent, h, k);
        }
    }
    __syncthreads();
    // clusters = connected components of the "boxes touch" graph; members of a cluster are written contiguously
    for (int h = tid; h < n_hot; h += nt) {
        cbox[4 * h] = 0x7fffffff; cbox[4 * h + 1] = 0x7fffffff; cbox[4 * h + 2] = -1; cbox[4 * h + 3] = 0;   // [3]: member count, then offset | count << 16
    }
    int* fill = (int*)idx_of;                           // per root (hot slot): members written so far
    int* ymax = fill + HOT_MAX;                         // per root: y1 of the bounding box
    for (int h = tid; h < n_hot; h += nt) { fill[h] = 0; ymax[h] = -1; }
    if (tid == 0) s_nroots = 0;
    __syncthreads();
    // bounding box per root: x0, y0, x1 in cbox[0..2], y1 in ymax[]; cbox[3] counts the members
    for (int h = tid; h < n_hot; h += nt) {
        if (box[4 * h] > box[4 * h + 2]) continue;
        int r = suf_find(parent, h);
        parent[h] = r;
        atomicMin(&cbox[4 * r], (int)tight[4 * h]); atomicMin(&cbox[4 * r + 1], (int)tight[4 * h + 1]);
        atomicMax(&cbox[4 * r + 2], (int)tight[4 * h + 2]); atomicMax(&ymax[r], (int)tight[4 * h + 3]);
        atomicAdd(&cbox[4 * r + 3], 1);
        if (r == h) { int k = atomicAdd(&s_nroots, 1); if (k < ROOTS_MAX) roots[k] = (uint16_t)h; }
    }
    __syncthreads();
    const int nr = s_nroots;
    if (nr > ROOTS_MAX) { if (tid == 0) cw.need_general[f] = 3; return; }
    // member offsets: exclusive scan of the counts over the root list (few hundred roots at most)
    if (tid == 0) {
        int acc = 0;
        for (int i = 0; i < nr; ++i) { int r = roots[i]; int c = cbox[4 * r + 3]; cbox[4 * r + 3] = acc | (c << 16); acc += c; }
    }
    __syncthreads();
    // member boxes of a cluster, contiguous from its offset (their order inside a cluster is irrelevant: ownership = "inside
    // any of them"); one thread per cluster sizes its bit rows and filter pieces.  The frame then reserves ONE contiguous
    // block of cluster ids, bit-row words and pieces (three global atomics per frame instead of three per cluster).
    short* memb = cw.memb + (size_t)f * HOT_MAX * 4;
    for (int h = tid; h < n_hot; h += nt) {
        if (box[4 * h] > box[4 * h + 2]) continue;
        const int r = parent[h];
        const int k = (cbox[4 * r + 3] & 0xffff) + atomicAdd(&fill[r], 1);
        *(uint2*)(memb + 4 * k) = *(const uint2*)(box + 4 * h);
    }
    for (int i = tid; i < nr; i += nt) {
        int r = roots[i];
        int y1 = ymax[r];
        int mw = cbox[4 * r + 2] - cbox[4 * r] + 1, mh = y1 - cbox[4 * r + 1] + 1;
        int pbx = cdiv_dev(mw, PIECE), pby = cdiv_dev(mh, PIECE);
        r_y1[i] = y1;
        r_words[i] = mh * pbx * (PIECE / 32);           // every piece owns whole words of the rows
        r_pcs[i] = pbx * pby;
    }
    __syncthreads();
    __shared__ int s_base[3];
    if (tid == 0) {
        unsigned tw = 0; int tp = 0;
        for (int i = 0; i < nr; ++i) {                  // exclusive prefixes, in place
            int w = r_words[i], pc = r_pcs[i];
            r_words[i] = (int)tw; r_pcs[i] = tp;
            tw += (unsigned)w; tp += pc;
        }
        int cid0 = atomicAdd(&cw.counters[CN_CLUSTERS], nr);
        unsigned roff0 = atomicAdd((unsigned*)&cw.counters[CN_ROWS], tw);
        int p00 = atomicAdd(&cw.counters[CN_PIECES], tp);
        s_base[0] = cid0; s_base[1] = (int)roff0; s_base[2] = p00;
        if (cid0 + nr > cw.cl_cap || roff0 + tw > cw.rows_cap || roff0 + tw < roff0 || p00 + tp > cw.pc_cap) s_bad = 1;
    }
    __syncthreads();
    const int cid0 = s_base[0], p00 = s_base[2];
    const unsigned roff0 = (unsigned)s_base[1];
    const bool bad = s_bad != 0;
    for (int i = tid; i < nr; i += nt) {
        int cid = cid0 + i;
        int r = roots[i];
        int x0 = cbox[4 * r], y0 = cbox[4 * r + 1], x1 = cbox[4 * r + 2], y1 = r_y1[i];
        int pbx = cdiv_dev(x1 - x0 + 1, PIECE), pby = cdiv_dev(y1 - y0 + 1, PIECE);
        int* ce = cw.clusters + 8 * (size_t)cid;
        if (bad) {                                       // (a cluster id beyond the table implies bad)
            if (cid < cw.cl_cap) { ce[0] = f; ce[1] = 1; ce[2] = 0; ce[3] = 0; ce[4] = 0; ce[5] = 0; }   // empty box: nothing downstream touches it
            for (int q = 0; q < pbx * pby; ++q) {        // the pieces this frame reserved become empty ones
                size_t pi = (size_t)p00 + (size_t)r_pcs[i] + (size_t)q;
                if (pi < (size_t)cw.pc_cap) { *(int4*)(cw.pieces + 8 * pi) = make_int4(0, 0, 0, 0); *(int4*)(cw.pieces + 8 * pi + 4) = make_int4(0, 0, 0, 0); }
            }
            continue;
        }
        ce[0] = f;
        ce[1] = x0 | (y0 << 16); ce[2] = x1 | (y1 << 16); ce[3] = (int)(roff0 + (unsigned)r_words[i]); ce[4] = pbx * (PIECE / 32);
        ce[5] = cbox[4 * r + 3]; ce[6] = 0; ce[7] = 0;
        for (int q = 0; q < pbx * pby; ++q)
            make_piece_desc(tv, f, lens, x0, y0, x1, y1, q % pbx, q / pbx, (unsigned)ce[3], ce[4], cw.pieces + 8 * (size_t)(p00 + r_pcs[i] + q));
    }
    if (tid == 0) {
        cw.frame_clusters[2 * f] = cid0; cw.frame_clusters[2 * f + 1] = bad ? 0 : nr;
        if (bad) cw.need_general[f] = 5;                // out of cluster / piece / bit-row storage: general path
    }
}

// ---------------------------------------------------------------------------------------------------------
// per piece: filter <= 64x64 output pixels of a cluster box in shared memory -> bit rows of the cluster (global)
// ---------------------------------------------------------------------------------------------------------
struct __align__(16) PieceSmem {
    static constexpr int UH = PIECE + 8, UW = PIECE + 12, BW = PIECE + 4, HSW = PIECE + 8;
    uint8_t U[UH * UW];            // undistorted pixels, origin (px0 - 4, py0 - 4); 0 outside the frame.  Row stride UW: the fast remap stores
                                   // quads aligned to frame columns that are multiples of 4, its rows start `lead` (0..3) pixels left of the box
    uint16_t HS[UH * HSW];         // horizontal 5-sums of U (U rows x B cols), rows 16-byte aligned
    uint8_t B[BW * BW];            // thresholded floor-mean, origin (px0 - 2, py0 - 2)
    // the horizontal 5-counts of B (B rows x output cols, BW * PIECE bytes) reuse U, which is dead by then; the packed path
    // keeps its bit planes in HS
};

__device__ __forceinline__ uint32_t maj3(uint32_t a, uint32_t b, uint32_t c) { return (a & b) | (c & (a | b)); }

// count of five 1-bit planes -> 3 bit planes (n0 + 2 n1 + 4 n2), 32 positions at a time
__device__ __forceinline__ void count5(uint32_t a, uint32_t b, uint32_t c, uint32_t d, uint32_t e, uint32_t& n0, uint32_t& n1, uint32_t& n2)
{
    uint32_t s1 = a ^ b ^ c, c1 = maj3(a, b, c);
    uint32_t s2 = s1 ^ d ^ e, c2 = maj3(s1, d, e);
    n0 = s2; n1 = c1 ^ c2; n2 = c1 & c2;
}

// Stages 2 and 3 of a piece that has no frame border within reach (count = 25, no clamping), packed:
//   A  horizontal 5-sums of U, four pixels per thread (two aligned 32-bit loads, sliding sum) -> HS (u16)
//   B  vertical 5-sums of HS, eight pixels per thread (128-bit loads, packed 16-bit adds and compare) -> one byte of the
//      thresholded bit row
//   C  bit-sliced 5x5 majority: per B row the horizontal 5-counts as three bit planes, per output row the sum of five
//      rows' planes (<= 25, five bit planes) and the test >= 13 -- 64 pixels per thread
// hl, hr, ht, hb (0 or 2): how far the thresholded-mean box extends beyond the piece on each side.  It stops at the
// cluster box: outside of it the thresholded mean cannot be set by this cluster's hot pixels (it would lie more than 2 from
// them), and whatever foreign hot pixels set there can only influence pixels that are not this cluster's foreground.
struct PackedDims { int mw, mh, hl, hr, ht, hb, lead; };   // lead: columns of U / HS / the bit rows left of the box (fast remap)

// ---- A ----  horizontal 5-sums of U -> HS
__device__ __forceinline__ void packed_stage_a(PieceSmem& S, const PackedDims& d)
{
    constexpr int UW = PieceSmem::UW, HSW = PieceSmem::HSW;
    const int tid = threadIdx.x;
    const int bw = d.mw + d.hl + d.hr + d.lead, uh = d.mh + d.ht + d.hb + 4;
    const int nq = (bw + 3) >> 2;
    const unsigned inv_q = (1u << 20) / (unsigned)nq + 1u;                        // t / nq == (t * inv_q) >> 20 (t * nq < 2^20)
    for (int t = tid; t < uh * nq; t += CL_THREADS) {
        int r = (int)(((unsigned)t * inv_q) >> 20), q = t - r * nq;
        const uint32_t* up = (const uint32_t*)&S.U[r * UW + 4 * q];
        uint32_t w0 = up[0], w1 = up[1];
#ifdef MOCAP_EMU
        uint32_t s0 = (w0 & 0xff) + ((w0 >> 8) & 0xff) + ((w0 >> 16) & 0xff) + (w0 >> 24) + (w1 & 0xff);
        uint32_t s1 = s0 - (w0 & 0xff) + ((w1 >> 8) & 0xff);
        uint32_t s2 = s1 - ((w0 >> 8) & 0xff) + ((w1 >> 16) & 0xff);
        uint32_t s3 = s2 - ((w0 >> 16) & 0xff) + (w1 >> 24);
#else
        // byte sums as dot products with 0/1 weights (IDP.4A): seven instructions for the four sums
        uint32_t s0 = __dp4a(w0, 0x01010101u, w1 & 0xffu);
        uint32_t s1 = __dp4a(w0, 0x01010100u, __dp4a(w1, 0x00000101u, 0u));
        uint32_t s2 = __dp4a(w0, 0x01010000u, __dp4a(w1, 0x00010101u, 0u));
        uint32_t s3 = __dp4a(w0, 0x01000000u, __dp4a(w1, 0x01010101u, 0u));
#endif
        uint2 v; v.x = s0 | (s1 << 16); v.y = s2 | (s3 << 16);
        *(uint2*)&S.HS[r * HSW + 4 * q] = v;
    }
}

// ---- B ----  bit rows of the thresholded mean: 16 bytes per row in S.B (72 bits used)
__device__ __forceinline__ void packed_stage_b(PieceSmem& S, const PackedDims& d, int T)
{
    constexpr int HSW = PieceSmem::HSW;
    const int tid = threadIdx.x;
    const int bw = d.mw + d.hl + d.hr + d.lead, bh = d.mh + d.ht + d.hb;
    uint8_t* bbits = S.B;
    const int no = (bw + 7) >> 3;
    const uint32_t bias = (0x8000u - (uint32_t)(25 * T)) * 0x00010001u;          // bit 15 of (v + bias) set  <=>  v >= 25 T
    // a thread keeps one column octet and walks down a segment of rows with a sliding 5-row sum: five 128-bit loads for its first
    // row, two (the row that enters, the row that leaves) for every further one
    // up to eight octets per row: a quarter warp per segment, so that the eight lanes whose 128-bit loads are served together read one
    // row's consecutive bytes (no bank conflict); the ninth octet of the widest boxes falls back to a dense numbering
    const int per = no <= 8 ? 8 : no;
    const unsigned inv_o = (1u << 16) / (unsigned)per + 1u;                       // t / per for t <= 128
    const int seg0 = (int)(((unsigned)tid * inv_o) >> 16), o = tid - seg0 * per;
    const int nseg = (int)(((unsigned)CL_THREADS * inv_o) >> 16);                 // row segments
    const int seg = o < no ? seg0 : nseg;                                         // surplus lanes idle
    const int rps = (bh + nseg - 1) / nseg;                                       // rows per segment
    const int r0 = seg * rps, r1 = min(bh, r0 + rps);
    if (seg < nseg && r0 < r1) {
        const uint16_t* hs = &S.HS[r0 * HSW + 8 * o];
        uint32_t a0 = 0, a1 = 0, a2 = 0, a3 = 0;
#pragma unroll
        for (int k = 0; k < 5; ++k) {
            const uint4 h = *(const uint4*)(hs + k * HSW);                        // one 128-bit load: eight sums
            a0 += h.x; a1 += h.y; a2 += h.z; a3 += h.w;                           // packed u16 adds: sums <= 6375, no carry across halves
        }
        for (int r = r0;;) {
            uint32_t m0 = (a0 + bias) & 0x80008000u, m1 = (a1 + bias) & 0x80008000u;
            uint32_t m2 = (a2 + bias) & 0x80008000u, m3 = (a3 + bias) & 0x80008000u;
            uint32_t y = (m0 >> 15) | (m1 >> 13) | (m2 >> 11) | (m3 >> 9);         // even bits 0..6 and 16..22
            bbits[r * 16 + o] = (uint8_t)((y & 0x55u) | ((y >> 15) & 0xAAu));
            if (++r >= r1) break;
            const uint4 hin = *(const uint4*)(hs + 5 * HSW), hout = *(const uint4*)hs;
            a0 += hin.x; a1 += hin.y; a2 += hin.z; a3 += hin.w;                   // the entering row first: no half ever borrows
            a0 -= hout.x; a1 -= hout.y; a2 -= hout.z; a3 -= hout.w;
            hs += HSW;
        }
    }
}

// ---- C1 ----  horizontal 5-counts per B row as three 64-bit planes (two 32-bit halves each), kept in S.HS (dead after B)
__device__ __forceinline__ void packed_stage_c1(PieceSmem& S, const PackedDims& d)
{
    const int tid = threadIdx.x;
    const int bw = d.mw + d.hl + d.hr, bh = d.mh + d.ht + d.hb;
    const uint8_t* bbits = S.B;
    uint32_t* planes = (uint32_t*)S.HS;                                           // [mh + 4][3][2]
    // plane row / bit position = offset from (piece - 2): the box rows and columns land at (2 - ht) / (2 - hl), what lies
    // outside the box is zero
    for (int r = tid; r < d.mh + 4; r += CL_THREADS) {
        const int rb = r - (2 - d.ht);
        uint32_t w0 = 0, w1 = 0, w2 = 0;
        if (rb >= 0 && rb < bh) {
            const uint32_t* bp = (const uint32_t*)&bbits[rb * 16];
            w0 = bp[0]; w1 = bp[1]; w2 = bp[2];                                   // bits 0..31, 32..63, 64..95
            if (d.lead) { w0 = __funnelshift_r(w0, w1, d.lead); w1 = __funnelshift_r(w1, w2, d.lead); w2 >>= d.lead; }   // drop the lead columns
            w2 &= 0xffu;
            if (bw < 32) { w0 &= (1u << bw) - 1u; w1 = 0; w2 = 0; }               // drop the surplus bits of the last byte
            else if (bw < 64) { w1 &= bw == 32 ? 0u : (1u << (bw - 32)) - 1u; w2 = 0; }
            else w2 &= bw == 64 ? 0u : (1u << (bw - 64)) - 1u;
            if (d.hl == 0) { w2 = (w2 << 2) | (w1 >> 30); w1 = (w1 << 2) | (w0 >> 30); w0 <<= 2; }
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            uint32_t lo = h ? w1 : w0, hi = h ? w2 : w1;
            uint32_t x1 = __funnelshift_r(lo, hi, 1), x2 = __funnelshift_r(lo, hi, 2), x3 = __funnelshift_r(lo, hi, 3), x4 = __funnelshift_r(lo, hi, 4);
            uint32_t n0, n1, n2;
            count5(lo, x1, x2, x3, x4, n0, n1, n2);
            planes[(r * 3 + 0) * 2 + h] = n0; planes[(r * 3 + 1) * 2 + h] = n1; planes[(r * 3 + 2) * 2 + h] = n2;
        }
    }
}

// ---- C2 ----  per output row: sum of five rows' counts (p + 2 q + 4 r with p, q, r = counts of the three planes) >= 13
__device__ __forceinline__ void packed_stage_c2(PieceSmem& S, const PackedDims& d, uint32_t* __restrict__ out, int wpr)
{
    const int tid = threadIdx.x;
    const uint32_t* planes = (const uint32_t*)S.HS;
    for (int t = tid; t < d.mh * 2; t += CL_THREADS) {
        int r = t >> 1, h = t & 1;
        uint32_t p0, p1, p2, q0, q1, q2, r0, r1, r2;
        const uint32_t* pl = planes + (size_t)r * 6 + h;
        count5(pl[0], pl[6], pl[12], pl[18], pl[24], p0, p1, p2);
        count5(pl[2], pl[8], pl[14], pl[20], pl[26], q0, q1, q2);
        count5(pl[4], pl[10], pl[16], pl[22], pl[28], r0, r1, r2);
        // total = p0 + 2 (p1 + q0) + 4 (p2 + q1 + r0) + 8 (q2 + r1) + 16 r2, rippled
        uint32_t b0 = p0;
        uint32_t b1 = p1 ^ q0, c1 = p1 & q0;
        uint32_t s2 = p2 ^ q1 ^ r0, c2 = maj3(p2, q1, r0);
        uint32_t b2 = s2 ^ c1, c2b = s2 & c1;
        uint32_t s3 = q2 ^ r1 ^ c2, c3 = maj3(q2, r1, c2);
        uint32_t b3 = s3 ^ c2b, c3b = s3 & c2b;
        uint32_t b4 = r2 | c3 | c3b;                                              // total <= 25: bit 5 cannot be set
        uint32_t ge13 = b4 | (b3 & b2 & (b1 | b0));
        int rem = d.mw - 32 * h;                                                  // keep only the piece's own columns
        if (rem < 32) ge13 &= rem > 0 ? ((1u << rem) - 1u) : 0u;
        out[(size_t)r * wpr + h] = ge13;
    }
}

// stages 2 and 3 of a piece with the frame border within reach: floor-mean of the in-frame taps > thresh (sum >= T * count),
// 5x5 majority with replicated frame border (clamped coordinates), bit rows via ballot
__device__ __forceinline__ void piece_threshold_majority(PieceSmem& S, int px0, int py0, int mw, int mh, int W, int H, int T,
                                                         uint32_t* __restrict__ out, int wpr)
{
    constexpr int BW = PieceSmem::BW, HSW = PieceSmem::HSW;
    uint8_t* MH = S.U;                                             // U is dead once HS is complete
    const int tid = threadIdx.x, lane = tid & 31, wy = tid >> 5, NWARP = CL_THREADS / 32;
    const int bw = mw + 4, bh = mh + 4;
    for (int r = wy; r < bh; r += NWARP) {
        int i = py0 - 2 + r;
        int cnty = min(i + 2, H - 1) - max(i - 2, 0) + 1;
        bool rowin = (unsigned)i < (unsigned)H;
        for (int c = lane; c < bw; c += 32) {
            int j = px0 - 2 + c, b = 0;
            if (rowin && (unsigned)j < (unsigned)W) {
                const uint16_t* h = &S.HS[r * HSW + c];
                int s = h[0] + h[HSW] + h[2 * HSW] + h[3 * HSW] + h[4 * HSW];
                int cnt = cnty * (min(j + 2, W - 1) - max(j - 2, 0) + 1);
                b = s >= T * cnt;
            }
            S.B[r * BW + c] = (uint8_t)b;
        }
        __syncwarp();
        const uint8_t* b = &S.B[r * BW] - (px0 - 2);                   // indexed by frame column
        for (int c = lane; c < mw; c += 32) {
            int j = px0 + c;
            MH[r * PIECE + c] = (uint8_t)(b[max(j - 2, 0)] + b[max(j - 1, 0)] + b[j] + b[min(j + 1, W - 1)] + b[min(j + 2, W - 1)]);
        }
    }
    __syncthreads();
    for (int r = wy; r < mh; r += NWARP) {
        int i = py0 + r;
        const int r0 = max(i - 2, 0) - (py0 - 2), r1 = max(i - 1, 0) - (py0 - 2), r2 = r + 2;
        const int r3 = min(i + 1, H - 1) - (py0 - 2), r4 = min(i + 2, H - 1) - (py0 - 2);
#pragma unroll
        for (int c0 = 0; c0 < PIECE; c0 += 32) {
            int c = c0 + lane, s = 0;
            if (c < mw) s = MH[r0 * PIECE + c] + MH[r1 * PIECE + c] + MH[r2 * PIECE + c] + MH[r3 * PIECE + c] + MH[r4 * PIECE + c];
            unsigned wv = __ballot_sync(0xffffffffu, s >= 13);
            if (lane == 0) out[(size_t)r * wpr + (c0 >> 5)] = wv;
        }
    }
}

// four fast-map words, kept in L2 (evict last: every piece of every frame reads the map, the frames stream past it)
// The L2 policies of the piece filter: the windows are read once (evict first), the fast map by every piece (PF_MAP_EVICT).  The
// kernel creates them where it uses them, once per piece: a 64-bit policy held across the piece loop costs it spills at 64 registers.
#ifdef MOCAP_EMU
static inline int4 ld_map4(const int32_t* p, uint64_t) { return *(const int4*)p; }
static inline uint64_t window_l2_policy() { return 0; }
static inline uint64_t map_l2_policy() { return 0; }
#else
__device__ __forceinline__ int4 ld_map4(const int32_t* p, uint64_t policy)
{
    int4 r;
    asm volatile("ld.global.nc.L2::cache_hint.v4.s32 {%0,%1,%2,%3}, [%4], %5;" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p), "l"(policy));
    return r;
}
#define PF_STR2(x) #x
#define PF_STR(x) PF_STR2(x)
__device__ __forceinline__ uint64_t window_l2_policy()
{
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t map_l2_policy()
{
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::" PF_STR(PF_MAP_EVICT) ".b64 %0, 1.0;" : "=l"(p));
    return p;
}
#endif

// one undistorted pixel from the staged window: m = fast-map word (fx | fy << 8 | tap offset << 16), p = the pixel's own place in the window
__device__ __forceinline__ uint32_t fast_tap(const uint8_t* p, uint32_t m)
{
    const uint8_t* q = p + ((int)m >> 16);
    const int fx = (int)(m & 0xffu), fy = (int)__byte_perm(m, 0, 0x4441);      // byte 1, one PRMT
    const int r0 = (32 - fx) * q[0] + fx * q[1];
    const int r1 = (32 - fx) * q[WIN_W] + fx * q[WIN_W + 1];
    return (uint32_t)(((32 - fy) * r0 + fy * r1 + 512) >> 10);
}

// work split of the fast remap: the quads of the U box (four pixels of a row each) as a flat index, thread t takes quads t, t + 128, ...:
// first quad (row r, quad column q), the step of 128 quads as (dr rows, dq quads) and the first map address
struct FastIter { int r, q, nq, dr, dq, uh; const int32_t* mp; bool on; };
__device__ __forceinline__ FastIter fast_iter_init(const int* d, const TableView& tv, int tid)
{
    const int px0 = d[1] & 0xffff, py0 = d[1] >> 16, dims = d[2];
    const int hl = (dims >> 16) & 3, hr = (dims >> 18) & 3, ht = (dims >> 20) & 3, hb = (dims >> 22) & 3;
    const int ux0 = px0 - hl - 2, lead = ux0 & 3;                              // quads are aligned to frame columns that are multiples of 4
    const int uw = (dims & 0xff) + hl + hr + 4 + lead;
    FastIter it;
    it.uh = ((dims >> 8) & 0xff) + ht + hb + 4;
    it.nq = (uw + 3) >> 2;                                                     // quads per row, <= 19
    const unsigned inv = (1u << 16) / (unsigned)it.nq + 1u;                    // t / nq == (t * inv) >> 16 for t <= 128
    it.on = ((dims >> 26) & 1) != 0;
    it.r = (int)(((unsigned)tid * inv) >> 16);
    it.q = tid - it.r * it.nq;
    it.dr = (int)(((unsigned)CL_THREADS * inv) >> 16);
    it.dq = CL_THREADS - it.dr * it.nq;
    it.mp = tv.fast + (size_t)d[6] * tv.lens_words + (size_t)(py0 - ht - 2 + it.r) * tv.W + (ux0 - lead) + 4 * it.q;
    return it;
}

// The source window of a piece comes in as ONE TMA box (cp.async.bulk.tensor.3d of the frame batch viewed as [n][H][W], WIN_W x
// WIN_H_LOW or WIN_W x WIN_H bytes at (wx0, wy0, frame); what lies outside the frame is zero-filled by the TMA unit), issued by thread
// 0 and completing on `wbar`.  Pieces whose window does not fit take their taps from global memory and post nothing.  Readers of
// the window wait on `wbar` and then pass a __syncthreads() that the issuing thread reaches after posting (the emulation build's
// synchronous box copy and no-op barrier rely on that).
__device__ __forceinline__ void post_piece_window(uint8_t* win, const int* d, const CUtensorMap& tmap, const CUtensorMap& tmap_low, uint64_t* wbar)
{
    if (threadIdx.x != 0 || !((d[2] >> 25) & 1)) return;
    const bool low = ((d[4] >> 16) & 0xff) <= WIN_H_LOW;                           // window rows needed
    mbar_expect_tx(wbar, WIN_W * (low ? WIN_H_LOW : WIN_H));
    tma_load_box(win, low ? &tmap_low : &tmap, (int)(int16_t)(d[5] & 0xffff), d[5] >> 16, d[0], wbar, window_l2_policy());
}

// Persistent CTAs over the piece list.  The loop is software-pipelined over pieces: as soon as the remap of piece i has
// consumed `win`, thread 0 posts the source window of piece i + 1 into it (it lands while the stages of piece i run), warp 0
// fetches the descriptor of piece i + 2 and thread 0 draws the index of piece i + 3 -- no descriptor, window or work-counter
// latency is waited for inside the loop.  use_window: the host encoded both window tensor maps (the batch is one a tensor map
// can describe) and T lies in 0..256; else every piece takes its taps from global memory.
__global__ void __launch_bounds__(CL_THREADS, 8) piece_filter_kernel(const uint8_t* __restrict__ frames, int64_t fstride, TableView tv, int thresh,
                                                                  ClusterWs cw, const __grid_constant__ CUtensorMap tmap,
                                                                  const __grid_constant__ CUtensorMap tmap_low, int use_window)
{
    __shared__ PieceSmem S;
    __align__(128) __shared__ uint8_t win[WIN_W * WIN_H];          // staged source window
    __shared__ uint64_t wbar;                                      // "window landed" barrier
    unsigned wphase = 0;
    if (threadIdx.x == 0 && use_window) {
        mbar_init(&wbar, 1);
        mbar_init_fence();
    }
    __align__(16) __shared__ int s_desc[2][8];
    __shared__ int s_next;
    constexpr int UW = PieceSmem::UW, HSW = PieceSmem::HSW;
    const int tid = threadIdx.x, lane = tid & 31, wy = tid >> 5, NWARP = CL_THREADS / 32;
    const int H = tv.H, W = tv.W, T = thresh + 1;
    const bool t_ok = T >= 0 && T <= 256;                          // thresholds the packed stages can represent
    const int total = min(cw.counters[CN_PIECES], cw.pc_cap);
    if (tid == 0) s_next = atomicAdd(&cw.counters[CN_PIECE_CUR], 1);
    __syncthreads();
    const int item = s_next;
    if (item >= total) return;
    if (tid < 8) s_desc[0][tid] = cw.pieces[8 * (size_t)item + tid];
    // three pieces deep: piece i is processed from s_desc[slot], warp 0 holds the descriptor of piece i + 1 in registers (dn),
    // thread 0 the index of piece i + 2 (next, an atomic in flight)
    int nx = 0, dn = 0, next = 0;
    if (wy == 0) {
        nx = __shfl_sync(0xffffffffu, lane == 0 ? atomicAdd(&cw.counters[CN_PIECE_CUR], 1) : 0, 0);
        if (lane < 8 && nx < total) dn = cw.pieces[8 * (size_t)nx + lane];
        if (lane == 0) next = atomicAdd(&cw.counters[CN_PIECE_CUR], 1);
    }
    __syncthreads();
    if (use_window) post_piece_window(win, s_desc[0], tmap, tmap_low, &wbar);
    int slot = 0;
    for (;;) {
        const int* d = s_desc[slot];
        const int f = d[0], px0 = d[1] & 0xffff, py0 = d[1] >> 16;
        const int dims = d[2];
        PackedDims pd;
        pd.mw = dims & 0xff; pd.mh = (dims >> 8) & 0xff;
        pd.hl = (dims >> 16) & 3; pd.hr = (dims >> 18) & 3; pd.ht = (dims >> 20) & 3; pd.hb = (dims >> 22) & 3;
        pd.lead = 0;
        const int mw = pd.mw, mh = pd.mh;
        const bool packed = ((dims >> 24) & 1) && t_ok;
        const bool staged = ((dims >> 25) & 1) && use_window;
        const bool fastp = ((dims >> 26) & 1) && use_window;
        const int wpr = d[4] & 0xffff;
        const int wx0 = (int)(int16_t)(d[5] & 0xffff), wy0 = d[5] >> 16;
        uint32_t* out = cw.rows_out + (unsigned)d[3];
        const int px1 = px0 + mw - 1, py1 = py0 + mh - 1;
        const int ux0 = packed ? px0 - pd.hl - 2 : px0 - 4, uy0 = packed ? py0 - pd.ht - 2 : py0 - 4;      // origin of the U box
        const int ux1 = packed ? px1 + pd.hr + 2 : px1 + 4, uy1 = packed ? py1 + pd.hb + 2 : py1 + 4;
        const int uw = ux1 - ux0 + 1, uh = uy1 - uy0 + 1, bw = mw + 4;
        const uint8_t* fr = frames + (size_t)f * fstride;
        if (staged) { mbar_wait(&wbar, wphase); wphase ^= 1; }
        __syncthreads();                                            // the window of this piece has landed; the other descriptor slot is free
        if (wy == 0 && lane < 8) s_desc[slot ^ 1][lane] = dn;
        if (tid == 0) s_next = nx;
        // ---- 1. undistorted pixels of the U box (zero outside the frame): the uw x uh box is walked as a flat index (all
        //         lanes busy whatever the box width), four pixels per thread per pass so that the map loads of a pass are
        //         in flight together; the bilinear taps come from the staged window. ----------------------------------------
        if (fastp) {
            // fast path: the box lies inside the frame, its source window is staged and every pixel has a fast-map entry (fx, fy and
            // the place of its first tap in the window relative to the pixel's own).  The box is cut into quads of four pixels aligned
            // to frame columns that are multiples of four, as a flat index; a thread takes every 128th quad (pointer steps with one wrap
            // test): ONE 128-bit load of the four map words (16-byte aligned: a quarter of the L1 requests of four 32-bit loads, the
            // kernel is bound by the L1 data pipe), sixteen byte taps from the window, one 32-bit store of the four results.  The pixels
            // left / right of the box in its first / last quad are real pixels (the descriptor's window and fast-map test cover them).
            // Measured and dropped: fetching the map words of the next quad (or of the first PF quads) ahead -- more loads in flight made
            // the kernel slower (0.82 -> 0.88-0.99 ms), the L1 pipe is the limit, not the L2 latency; four pixels of a COLUMN per thread
            // (the byte taps of a warp then fall into consecutive bytes: no 2-way bank conflicts, but four 32-bit map loads and four byte
            // stores): 0.680 against 0.687 ms, and no gain with two calls in flight.
            FastIter fi = fast_iter_init(d, tv, tid);
            const uint64_t mpolicy = map_l2_policy();
            pd.lead = ux0 & 3;
            const uint8_t* pw = win + (uy0 - wy0 + fi.r) * WIN_W + (ux0 - pd.lead - wx0) + 4 * fi.q;
            uint8_t* pu = S.U + fi.r * UW + 4 * fi.q;
            const int dw = fi.dr * WIN_W + 4 * fi.dq, du = fi.dr * UW + 4 * fi.dq, dm = fi.dr * W + 4 * fi.dq;
            const int dwx = WIN_W - 4 * fi.nq, dux = UW - 4 * fi.nq, dmx = W - 4 * fi.nq;          // the wrap into the next row
            while (fi.r < uh) {
                const int4 m = ld_map4(fi.mp, mpolicy);                          // 16-byte aligned: W, the table and the quad column are
                *(uint32_t*)pu = fast_tap(pw, (uint32_t)m.x) | (fast_tap(pw + 1, (uint32_t)m.y) << 8) | (fast_tap(pw + 2, (uint32_t)m.z) << 16) |
                                 (fast_tap(pw + 3, (uint32_t)m.w) << 24);
                fi.q += fi.dq; fi.r += fi.dr; fi.mp += dm; pw += dw; pu += du;
                if (fi.q >= fi.nq) { fi.q -= fi.nq; ++fi.r; fi.mp += dmx; pw += dwx; pu += dux; }
            }
        } else {
            const int32_t* map = tv.map + (size_t)d[6] * tv.lens_words;
            const int n_u = uw * uh;
            const unsigned inv = (1u << 20) / (unsigned)uw + 1u;              // idx / uw == (idx * inv) >> 20 for idx * uw < 2^20
            for (int base = tid; base < n_u; base += 4 * CL_THREADS) {
                uint32_t m[4]; int ii[4], jj[4], rc[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    int idx = base + k * CL_THREADS;
                    int r = (int)(((unsigned)idx * inv) >> 20), c = idx - r * uw;
                    int i = uy0 + r, j = ux0 + c;
                    ii[k] = i; jj[k] = j; rc[k] = r * UW + c;
                    m[k] = (idx < n_u && (unsigned)i < (unsigned)H && (unsigned)j < (unsigned)W) ? (uint32_t)map[(size_t)i * W + j] : MAP_OUTSIDE;
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    int val = 0;
                    uint32_t mm = m[k];
                    if (staged) {
                        if (mm != MAP_OUTSIDE) {
                            int iu = 32 * jj[k] + (int)(int16_t)(mm & 0xffff);
                            int iv = 32 * ii[k] + (int)(int16_t)(mm >> 16);
                            int fx = iu & 31, fy = iv & 31;
                            const uint8_t* p = &win[((iv >> 5) - wy0) * WIN_W + ((iu >> 5) - wx0)];
                            int r0 = (32 - fx) * p[0] + fx * p[1];
                            int r1 = (32 - fx) * p[WIN_W] + fx * p[WIN_W + 1];
                            val = ((32 - fy) * r0 + fy * r1 + 512) >> 10;
                        }
                    } else {
                        val = remap_px(fr, W, H, ii[k], jj[k], mm);
                    }
                    if (base + k * CL_THREADS < n_u) S.U[rc[k]] = (uint8_t)val;
                }
            }
        }
        __syncthreads();                                            // U complete; the window is free again
        // post the next piece's window (it lands while the stages below run), fetch the descriptor of the piece after it
        if (s_next < total && use_window) post_piece_window(win, s_desc[slot ^ 1], tmap, tmap_low, &wbar);
        if (wy == 0) {
            nx = __shfl_sync(0xffffffffu, next, 0);
            dn = (lane < 8 && nx < total) ? cw.pieces[8 * (size_t)nx + lane] : 0;
            if (lane == 0) next = atomicAdd(&cw.counters[CN_PIECE_CUR], 1);
        }
        if (packed) {
            packed_stage_a(S, pd);
            __syncthreads();
            packed_stage_b(S, pd, T);
            __syncthreads();
            packed_stage_c1(S, pd);
            __syncthreads();
            packed_stage_c2(S, pd, out, wpr);
        } else {
            // plain per-pixel stages with the full +-4 halo and clamped coordinates (frame border within reach)
            for (int r = wy; r < uh; r += NWARP)
                for (int c = lane; c < bw; c += 32) {
                    const uint8_t* up = &S.U[r * UW + c];
                    S.HS[r * HSW + c] = (uint16_t)(up[0] + up[1] + up[2] + up[3] + up[4]);
                }
            __syncthreads();
            piece_threshold_majority(S, px0, py0, mw, mh, W, H, T, out, wpr);
        }
        if (s_next >= total) break;
        slot ^= 1;
    }
}

// ---------------------------------------------------------------------------------------------------------
// per cluster row: border-start candidates.  A run with no 8-neighbour above starts an outer border, a gap between two
// runs that is completely covered from above starts a hole border (necessary conditions; the trace verifies them).
// Only candidates the cluster owns are kept: start pixel inside one of its own cell boxes.
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void emit_candidate(const ClusterWs& cw, int cid, int f, const short* memb, int m_cnt, int cx, int r, int cty, int cx0, int cy0)
{
    int ax = cx + cx0, ay = r + cy0;
    bool own = false;
    for (int m = 0; m < m_cnt && !own; ++m)
        own = ax >= memb[4 * m] && ax <= memb[4 * m + 2] && ay >= memb[4 * m + 1] && ay <= memb[4 * m + 3];
    if (!own) return;
    int slot = atomicAdd(&cw.cand_count[f], 1);              // per-frame lists: no single hot counter
    if (slot >= CAND_PER_FRAME) { cw.need_general[f] = 7; return; }
    int* e = cw.cand_list + 2 * ((size_t)f * CAND_PER_FRAME + slot);
    e[0] = cid;
    e[1] = cx | (r << 16) | (cty << 31);
}

// first bit >= x that differs from `inv` (inv = 0: first set bit, inv = ~0: first clear bit); wpr * 32 if none
__device__ __forceinline__ int next_bit(const uint32_t* row, int wpr, int x, uint32_t inv)
{
    int wi = x >> 5;
    uint32_t w = (row[wi] ^ inv) & (~0u << (x & 31));
    while (!w && ++wi < wpr) w = row[wi] ^ inv;
    return w ? wi * 32 + __ffs(w) - 1 : wpr * 32;
}
__device__ __forceinline__ uint32_t range_mask(int wi, int lo, int hi)          // bits of word wi inside [lo, hi]
{
    int a = max(lo - wi * 32, 0), b = min(hi - wi * 32, 31);
    return (b == 31 ? ~0u : ((1u << (b + 1)) - 1u)) & (~0u << a);
}
__device__ __forceinline__ bool range_any(const uint32_t* row, int lo, int hi)
{
    for (int wi = lo >> 5; wi <= (hi >> 5); ++wi) if (row[wi] & range_mask(wi, lo, hi)) return true;
    return false;
}
__device__ __forceinline__ bool range_all(const uint32_t* row, int lo, int hi)   // empty range: true
{
    if (lo > hi) return true;
    for (int wi = lo >> 5; wi <= (hi >> 5); ++wi) { uint32_t m = range_mask(wi, lo, hi); if ((row[wi] & m) != m) return false; }
    return true;
}

__global__ void __launch_bounds__(128) candidates_kernel(ClusterWs cw)
{
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
    const int total = min(cw.counters[CN_CLUSTERS], cw.cl_cap);
    // the cluster entry of the warp's next cluster is fetched while the current one is scanned
    int4 ea = make_int4(0, 0, 0, 0), eb = ea;
    if (warp < total) { ea = *(const int4*)(cw.clusters + 8 * (size_t)warp); eb = *(const int4*)(cw.clusters + 8 * (size_t)warp + 4); }
    for (int cid = warp; cid < total; cid += nwarps) {
        const int4 ca = ea, cb = eb;
        if (cid + nwarps < total) {
            ea = *(const int4*)(cw.clusters + 8 * (size_t)(cid + nwarps)); eb = *(const int4*)(cw.clusters + 8 * (size_t)(cid + nwarps) + 4);
        }
        const int f = ca.x;
        const int cx0 = ca.y & 0xffff, cy0 = ca.y >> 16, cx1 = ca.z & 0xffff, cy1 = ca.z >> 16, wpr = cb.x;
        const int mw = cx1 - cx0 + 1, mh = cy1 - cy0 + 1;
        if (mw <= 0 || cw.need_general[f]) continue;
        const int m_off = cb.y & 0xffff, m_cnt = cb.y >> 16;
        const short* memb = cw.memb + ((size_t)f * HOT_MAX + m_off) * 4;
        const uint32_t* rows = cw.rows_out + (unsigned)ca.w;
        for (int r = lane; r < mh; r += 32) {
            const uint32_t* row = rows + (size_t)r * wpr;
            if (wpr == 2) {
                // box at most 64 wide: the row and the row above are one 64-bit word each, runs and gaps come from bit scans
                // (bit-row storage is handed out in even word counts, so these rows are 8-byte aligned)
                unsigned long long cur = *(const unsigned long long*)row, up = 0ull;
                if (r > 0) up = *(const unsigned long long*)(row - 2);
                int last_end = -2;
                while (cur) {
                    int s0 = __ffsll((long long)cur) - 1;
                    unsigned long long t = cur >> s0;
                    int len = (~t) ? __ffsll((long long)~t) - 1 : 64;
                    unsigned long long runmask = (len >= 64 ? ~0ull : ((1ull << len) - 1ull)) << s0;
                    cur &= ~runmask;
                    int e0 = s0 + len - 1;
                    unsigned long long dil = runmask | (runmask << 1) | (runmask >> 1);
                    if (last_end >= 0 && r > 0) {
                        unsigned long long gap = ((1ull << s0) - 1ull) & ~((2ull << last_end) - 1ull);      // bits last_end+1 .. s0-1
                        if ((up & gap) == gap) emit_candidate(cw, cid, f, memb, m_cnt, last_end, r, 1, cx0, cy0);
                    }
                    if ((up & dil) == 0ull) emit_candidate(cw, cid, f, memb, m_cnt, s0, r, 0, cx0, cy0);
                    last_end = e0;
                }
                continue;
            }
            // wider boxes: the same run / gap logic with word scans (bits at x >= mw are zero in every row)
            const uint32_t* above = row - wpr;
            int x = 0, last_end = -2;
            while (x < mw) {
                int s0 = next_bit(row, wpr, x, 0u);
                if (s0 >= mw) break;
                int e1 = min(next_bit(row, wpr, s0, ~0u), mw);              // first clear bit after the run
                if (last_end >= 0 && r > 0 && range_all(above, last_end + 1, s0 - 1))
                    emit_candidate(cw, cid, f, memb, m_cnt, last_end, r, 1, cx0, cy0);
                if (r == 0 || !range_any(above, max(s0 - 1, 0), min(e1, mw - 1)))
                    emit_candidate(cw, cid, f, memb, m_cnt, s0, r, 0, cx0, cy0);
                last_end = e1 - 1;
                x = e1;
            }
        }
    }
}

// Start pixel (frame index) of the outer border of the blob that owns the hole border starting at local pixel (lx, ly):
// the west edge of the leftmost pixel of that pixel's run lies on another border of the same blob; if that border's
// smallest edge is a west edge it is the blob's outer border, otherwise it is another hole of the blob further left and the
// search continues from there.  -1 if it does not settle.  The box: mw x mh pixels at (ox, oy) of a frame Wabs wide.
__device__ long long hole_parent_start(const uint32_t* rows, int mw, int mh, int wpr, int lx, int ly, int ox, int oy, int Wabs, int* overflow)
{
    for (int hop = 0; hop < 32; ++hop) {
        const uint32_t* row = rows + (size_t)ly * wpr;
        int x = lx;
        while (x > 0 && ((row[(x - 1) >> 5] >> ((x - 1) & 31)) & 1u)) --x;     // leftmost pixel of the run
        long long a[3], mk; double per; int nch;
        trace_border<true, true>(rows, mh, wpr, mw, x, ly, 4, -1, a, &per, &nch, overflow, ox, oy, Wabs, nullptr, &mk);
        if (*overflow) return -1;
        const long long pix = mk >> 1;                             // smallest edge of the border through that west edge
        if ((mk & 1) == 0) return pix;
        ly = (int)(pix / Wabs) - oy; lx = (int)(pix % Wabs) - ox;  // start pixel of another hole border of the same blob
    }
    return -1;
}

// One CTA per frame, one thread per owned border-start candidate: Suzuki-Abe trace on the cluster's bit rows.  A completed
// border becomes a record of its frame; hole borders also record their blob's outer border (their parent in the contour
// tree).  Afterwards the frame is checked for nesting (an outer border starting inside the bounding box of a hole border):
// only then the contour tree is deeper than outer -> hole and the frame goes to the general path.
__device__ void frame_traces(const ClusterWs& cw, int f, int W, int max_contours)
{
    __shared__ int s_holes;
    if (threadIdx.x == 0) s_holes = 0;
    __syncthreads();
    const int n_cand = min(cw.cand_count[f], CAND_PER_FRAME);
    // Work order: a warp traces 32 borders in lockstep, so its time is its longest border.  The candidates are therefore
    // counting-sorted by the size of their cluster box (a proxy for the border length), longest first: the boxes wider than
    // 64 pixels (several blobs next to each other) or higher than 1024, traced on a sliding 64-pixel window, then, from a
    // warp boundary, the other boxes up to 64 wide (one 64-bit load per row).  A second pass
    // over the list runs in reverse thread order, so that the shortest borders follow the shortest first-pass borders.
    __shared__ uint16_t s_order[CAND_PER_FRAME + 32];          // + the padding between the two lists
    __shared__ int s_bucket[34];
    if (threadIdx.x < 34) s_bucket[threadIdx.x] = 0;
    __syncthreads();
    auto bucket_of = [&](const int* ce) -> int {
        int mw = (ce[2] & 0xffff) - (ce[1] & 0xffff) + 1, mh = (ce[2] >> 16) - (ce[1] >> 16) + 1;
        bool narrow = ce[4] == 2 && mh <= 1024;
        int b = 15 - min((mw + mh) >> 4, 15);
        return narrow ? 16 + b : b;
    };
    for (int cslot = threadIdx.x; cslot < n_cand; cslot += blockDim.x)
        atomicAdd(&s_bucket[1 + bucket_of(cw.clusters + 8 * (size_t)cw.cand_list[2 * ((size_t)f * CAND_PER_FRAME + cslot)])], 1);
    __syncthreads();
    if (threadIdx.x == 0) {
        int acc = 0;
        for (int b = 1; b <= 32; ++b) { int c = s_bucket[b]; s_bucket[b] = acc; acc += c; if (b == 16) { s_bucket[33] = acc; acc = (acc + 31) & ~31; } }
        // s_bucket[1 + b] = start of bucket b; the narrow buckets (16..31) start on a warp boundary; s_bucket[33] = #wide
        s_bucket[0] = acc;                                       // padded total
    }
    __syncthreads();
    const int n_wide = s_bucket[33], n_pad = (n_wide + 31) & ~31, n_total = s_bucket[0];
    for (int i = threadIdx.x; i < CAND_PER_FRAME + 32; i += blockDim.x) s_order[i] = 0xffff;
    __syncthreads();
    for (int cslot = threadIdx.x; cslot < n_cand; cslot += blockDim.x) {
        int b = bucket_of(cw.clusters + 8 * (size_t)cw.cand_list[2 * ((size_t)f * CAND_PER_FRAME + cslot)]);
        int pos = atomicAdd(&s_bucket[1 + b], 1);
        s_order[pos] = (uint16_t)cslot;                          // pos < n_cand + 31 <= CAND_PER_FRAME + 31
    }
    __syncthreads();
    for (int base = 0, pass = 0; base < n_total; base += blockDim.x, ++pass) {
        const int it = base + ((pass & 1) ? (int)(blockDim.x - 1 - threadIdx.x) : (int)threadIdx.x);
        if (it >= n_total) continue;
        const int cslot = s_order[it];
        if (cslot == 0xffff) continue;                           // padding between the two lists
        const size_t c = (size_t)f * CAND_PER_FRAME + cslot;
        const int* ce = cw.clusters + 8 * (size_t)cw.cand_list[2 * c];
        const int code = cw.cand_list[2 * c + 1];
        const int mx0 = ce[1] & 0xffff, my0 = ce[1] >> 16, mx1 = ce[2] & 0xffff, my1 = ce[2] >> 16;
        const int lx = code & 0xffff, ly = (code >> 16) & 0x7fff, ty = (code >> 31) & 1;
        const uint32_t* rows = cw.rows_out + (unsigned)ce[3];
        const int mw = mx1 - mx0 + 1, mh = my1 - my0 + 1, wpr = ce[4];
        long long st = (long long)(ly + my0) * W + (lx + mx0);
        long long a[3]; double per; int nch, ovf = 0, bbox[4];
        int ok;
        if (it >= n_pad) ok = trace_border<false>(rows, mh, 2, mw, lx, ly, ty ? 0 : 4, 2 * st + ty, a, &per, &nch, &ovf, mx0, my0, W, bbox);
        else ok = trace_border<true>(rows, mh, wpr, mw, lx, ly, ty ? 0 : 4, 2 * st + ty, a, &per, &nch, &ovf, mx0, my0, W, bbox);
        if (ovf) { cw.need_general[f] = 8; continue; }
        if (!ok) continue;
        long long parent = -1;
        if (ty) {
            parent = hole_parent_start(rows, mw, mh, wpr, lx, ly, mx0, my0, W, &ovf);
            if (parent < 0) { cw.need_general[f] = 8; continue; }
            atomicAdd(&s_holes, 1);
        }
        int slot = atomicAdd(&cw.rec_count[f], 1);
        if (slot < max_contours) {
            size_t k = (size_t)f * max_contours + slot;
            cw.rec_start[k] = (int)st;
            long long* ra = cw.rec_a + k * 3;
            ra[0] = a[0]; ra[1] = a[1]; ra[2] = a[2];
            cw.rec_per[k] = per;
            int* ri = cw.rec_info + k * 4;
            ri[0] = ty; ri[1] = (int)parent; ri[2] = bbox[0] | (bbox[1] << 16); ri[3] = bbox[2] | (bbox[3] << 16);
        }
    }
    __syncthreads();
    if (s_holes == 0) return;
    // nesting check: an outer border whose start pixel lies inside the bounding box of a hole border
    const int n = min(cw.rec_count[f], max_contours);
    const int* start = cw.rec_start + (size_t)f * max_contours;
    const int* info = cw.rec_info + (size_t)f * max_contours * 4;
    for (int h = threadIdx.x; h < n; h += blockDim.x) {
        if (!info[4 * h]) continue;
        int x0 = info[4 * h + 2] & 0xffff, y0 = info[4 * h + 2] >> 16, x1 = info[4 * h + 3] & 0xffff, y1 = info[4 * h + 3] >> 16;
        for (int o = 0; o < n; ++o) {
            if (info[4 * o]) continue;
            int ox = start[o] % W, oy = start[o] / W;
            if (ox > x0 && ox < x1 && oy > y0 && oy < y1) { cw.need_general[f] = 9; break; }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// per frame: the reference's filter, centroid and output order on the frame's border records
// ---------------------------------------------------------------------------------------------------------
__device__ void frame_finalize(const ClusterWs& cw, int f, uint8_t* keepv /*[max_contours], shared*/, int max_contours, int max_blobs,
                               double min_area, double min_circ,
                               int32_t* __restrict__ out_xy, int xy_float, int32_t* __restrict__ out_count, int32_t* __restrict__ out_flags,
                               double* __restrict__ out_contours, int32_t* __restrict__ out_contour_count)
{
    const int tid = threadIdx.x;
    const int n = cw.rec_count[f];
    __shared__ int s_kept;
    if (tid == 0) s_kept = 0;
    __syncthreads();
    if (n > max_contours) {
        if (tid == 0) { out_flags[f] |= MOCAP_FLAG_CONTOUR_OVERFLOW; out_count[f] = 0; if (out_contour_count) out_contour_count[f] = 0; }
        return;
    }
    const int* start = cw.rec_start + (size_t)f * max_contours;
    const long long* ra = cw.rec_a + (size_t)f * max_contours * 3;
    const double* rper = cw.rec_per + (size_t)f * max_contours;
    const int* info = cw.rec_info + (size_t)f * max_contours * 4;
    for (int c = tid; c < n; c += (int)blockDim.x) keepv[c] = (uint8_t)contour_keep(ra[3 * c], rper[c], min_area, min_circ);
    __syncthreads();
    for (int c = tid; c < n; c += (int)blockDim.x) {
        long long a00 = ra[3 * c], a10 = ra[3 * c + 1], a01 = ra[3 * c + 2];
        double per = rper[c];
        int keep = keepv[c];
        // cv.findContours order for a two-level tree (top-level outer borders, each followed by its hole borders): outer
        // borders in reverse raster order of their start pixel, the holes of a blob in reverse raster order of theirs
        const int hole = info[4 * c], st = start[c];
        const int top = hole ? info[4 * c + 1] : st;          // start pixel of the top-level border of my subtree
        int rank = 0, pos = 0, parent_rank = -1;
        for (int u = 0; u < n; ++u) {
            const int uh = info[4 * u], us = start[u], ut = uh ? info[4 * u + 1] : us;
            bool before;
            if (ut != top) before = ut > top;                 // another blob's subtree
            else if (uh != hole) before = !uh;                // my blob: the outer border first
            else before = us > st;                            // sibling holes
            rank += before;
            pos += before && keepv[u];
        }
        if (hole) {                                           // rank of my parent = number of subtrees that start later
            parent_rank = 0;
            for (int u = 0; u < n; ++u) {
                const int uh = info[4 * u], us = start[u], ut = uh ? info[4 * u + 1] : us;
                parent_rank += ut > top;
            }
        }
        if (out_contours && rank < max_contours) {
            double* o = out_contours + ((size_t)f * max_contours + rank) * 8;
            o[0] = (double)a00; o[1] = (double)a10; o[2] = (double)a01; o[3] = per;
            o[4] = (double)hole; o[5] = (double)parent_rank; o[6] = (double)keep; o[7] = (double)st;
        }
        if (!keep) continue;
        atomicAdd(&s_kept, 1);
        if (pos < max_blobs) store_blob_centroid(out_xy + ((size_t)f * max_blobs + pos) * 2, a00, a10, a01, xy_float);
    }
    __syncthreads();
    if (tid == 0) {
        int kept = s_kept;
        if (kept > max_blobs) { out_flags[f] |= MOCAP_FLAG_BLOB_OVERFLOW; kept = max_blobs; }
        out_count[f] = kept;
        if (out_contour_count) out_contour_count[f] = n;
    }
}

// One CTA per frame: the traces of the frame's border-start candidates, the nesting check and -- unless the frame was
// handed to the general path on the way -- the reference's filter / centroid / output order.
__global__ void __launch_bounds__(CL_THREADS, BORDERS_MIN_CTAS) borders_finalize_kernel(ClusterWs cw, int W, int frame_step, int max_contours, int max_blobs, double min_area, double min_circ,
                                                                      int32_t* __restrict__ out_xy, int xy_float, int32_t* __restrict__ out_count, int32_t* __restrict__ out_flags,
                                                                      double* __restrict__ out_contours, int32_t* __restrict__ out_contour_count)
{
    DYN_SHARED(smraw);
    // CTA b takes frame b * frame_step mod n (frame_step coprime to n): consecutive frames of a batch come from the same
    // cameras in the same order, so a plain b -> frame map would hand every SM frames of the same few cameras
    const int f = (int)(((long long)blockIdx.x * frame_step) % cw.n_frames);
    if (cw.need_general[f]) return;
    step_table_build();                                     // (frame_traces synchronises before its traces)
    frame_traces(cw, f, W, max_contours);
    __syncthreads();
    if (cw.need_general[f]) return;                         // trace budget, unresolved hole parent or nested contour tree
    frame_finalize(cw, f, (uint8_t*)smraw, max_contours, max_blobs, min_area, min_circ, out_xy, xy_float, out_count, out_flags, out_contours, out_contour_count);
}

// ---------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------
static int cl_cap_of(int n) { return n * 256 + 1024; }
static int pc_cap_of(int n) { return n * 512 + 2048; }
static size_t rows_cap_of(int n, int H, int W) { size_t w = (size_t)n * ((size_t)H * W / 128 + 4096); return w > 0xf0000000ull ? 0xf0000000ull : w; }   // a quarter of the frame area per frame

size_t cluster_ws_bytes(int n, int H, int W, int max_contours, ClusterLayout* L)
{
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t r = off; off += align_up(bytes, 256); return r; };
    L->counters = take(64);
    L->rec_count = take((size_t)n * 4);
    L->cand_count = take((size_t)n * 4);
    L->frame_clusters = take((size_t)n * 8);
    L->zero_bytes = off;
    L->clusters = take((size_t)cl_cap_of(n) * 32);
    L->pieces = take((size_t)pc_cap_of(n) * 32);
    L->rec_start = take((size_t)n * max_contours * 4);
    L->rec_a = take((size_t)n * max_contours * 24);
    L->rec_per = take((size_t)n * max_contours * 8);
    L->memb = take((size_t)n * HOT_MAX * 8);
    L->rows_out = take(rows_cap_of(n, H, W) * 4);
    L->cand_list = take((size_t)n * CAND_PER_FRAME * 8);
    L->rec_info = take((size_t)n * max_contours * 16);
    return off;
}

bool cluster_path_supported(int H, int W)
{
    return cdiv(W, TILE) * cdiv(H, TILE) <= CELLS_MAX && W <= 32767 && H <= 32767;
}

int launch_cluster_path(const uint8_t* frames, int n, int H, int W, int64_t fstride, const TableView& tv, int thresh,
                        const uint32_t* cellbox, char* ws_base, const ClusterLayout& L, int* need_general,
                        int max_contours, int max_blobs, double min_area, double min_circ,
                        int32_t* out_xy, int xy_float, int32_t* out_count, int32_t* out_flags, double* out_contours, int32_t* out_contour_count,
                        cudaStream_t s, StageTimer* timer, const ClusterLaunch& how)
{
    ClusterWs cw;
    cw.need_general = need_general;
    cw.counters = (int*)(ws_base + L.counters);
    cw.clusters = (int*)(ws_base + L.clusters);
    cw.pieces = (int*)(ws_base + L.pieces);
    cw.cl_cap = cl_cap_of(n); cw.pc_cap = pc_cap_of(n);
    cw.rec_count = (int*)(ws_base + L.rec_count);
    cw.rec_start = (int*)(ws_base + L.rec_start);
    cw.rec_a = (long long*)(ws_base + L.rec_a);
    cw.rec_per = (double*)(ws_base + L.rec_per);
    cw.memb = (short*)(ws_base + L.memb);
    cw.rows_out = (uint32_t*)(ws_base + L.rows_out);
    cw.rows_cap = (unsigned)rows_cap_of(n, H, W);
    cw.cand_list = (int*)(ws_base + L.cand_list);
    cw.cand_count = (int*)(ws_base + L.cand_count);
    cw.rec_info = (int*)(ws_base + L.rec_info);
    cw.frame_clusters = (int*)(ws_base + L.frame_clusters);
    cw.n_frames = n;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int cells = tv.TX * tv.TY;
    size_t sm_form = (size_t)form_idx_slots(cells) * 2 + (size_t)HOT_MAX * (2 + 4 + 16 + 8 + 8) + (size_t)ROOTS_MAX * (2 + 12) + 64;
#ifndef MOCAP_EMU
    static bool attr_done = false;                          // (idempotent; a race only repeats the call)
    if (!attr_done) { CUDA_TRY(cudaFuncSetAttribute(form_clusters_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024)); attr_done = true; }
#endif
    stage_begin(timer, 1, s);
    LAUNCH(form_clusters_kernel, n, CL_THREADS, sm_form, s, cellbox, tv, cw, out_flags);
    stage_end(timer, 1, s);
    if (how.ev_group) cudaEventRecord(how.ev_group, s);
    stage_begin(timer, 2, s);
    {
        CUtensorMap tmap, tmap_low;
        memset(&tmap, 0, sizeof(tmap)); memset(&tmap_low, 0, sizeof(tmap_low));
        const int T = thresh + 1;
        const int use_window = (T >= 0 && T <= 256 && frames_tensor_map(&tmap, frames, n, H, W, fstride, WIN_W, WIN_H, PF_WIN_L2_PROMO) &&
                                frames_tensor_map(&tmap_low, frames, n, H, W, fstride, WIN_W, WIN_H_LOW, PF_WIN_L2_PROMO)) ? 1 : 0;
        LAUNCH(piece_filter_kernel, sms * how.filter_ctas, CL_THREADS, 0, s, frames, fstride, tv, thresh, cw, tmap, tmap_low, use_window);
    }
    stage_end(timer, 2, s);
    if (how.ev_filter) cudaEventRecord(how.ev_filter, s);
    stage_begin(timer, 3, s);
    LAUNCH(candidates_kernel, sms * how.cand_ctas, 128, 0, s, cw);
    int frame_step = 1;
    for (int pr : {61, 67, 71, 73}) if (n % pr != 0) { frame_step = pr; break; }          // a prime that does not divide n
    LAUNCH(borders_finalize_kernel, n, BF_THREADS, (size_t)max_contours + 16, s, cw, W, frame_step, max_contours, max_blobs, min_area, min_circ,
           out_xy, xy_float, out_count, out_flags, out_contours, out_contour_count);
    stage_end(timer, 3, s);
    if (how.ev_borders) cudaEventRecord(how.ev_borders, s);
    CUDA_TRY(cudaGetLastError());
    return MOCAP_OK;
}
