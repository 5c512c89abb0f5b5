// Suzuki-Abe border following on a packed binary image: one walker, trace_border, for every border of the library -- the
// per-cluster traces and hole-parent walks (detect_cluster.cu), the general path's traces, canonical-start tests and
// parent walks, and the outline of drawContours (detect_blobs.cu).  Restates what cv.findContours(RETR_TREE,
// CHAIN_APPROX_SIMPLE) does per border (lib/ImageOperations.py:41) plus the Green sums / perimeter of cv.moments /
// cv.arcLength (:44-45, :59).  A step is one byte of a step table in shared memory, looked up with the walker's 3x3
// neighbourhood taken from bit rows held in registers.
#pragma once
#include "common.cuh"

// The rule of one step: counter-clockwise search of the 8-neighbour mask m from s + 1 (s = direction to the previous
// pixel); returns the step direction, `zeros` = bitmask of neighbour directions examined and found empty.
__device__ __forceinline__ int walk_rule(uint32_t m, int s, unsigned& zeros)
{
    int start = (s + 1) & 7;
    uint32_t rot = ((m | (m << 8)) >> start) & 0xffu;             // bit k = m[(start + k) & 7]
    int k = rot ? __ffs(rot) - 1 : 8;
    uint32_t z = ((1u << k) - 1u) << start;                       // the k empty directions passed over
    zeros = (z | (z >> 8)) & 0xffu;
    return (start + k) & 7;
}

#define WALK_BUDGET (1 << 22)

// Step table of trace_border: walk_rule's outcome for every 3x3 neighbourhood and every s, so that a step is one
// shared-memory byte instead of gathering eight neighbour bits and searching them.  Index (raw9 << 3) + s, where raw9 is
// the walker's 3x3 neighbourhood as three row triples side by side: bits 0-2 the row above (columns x-1, x, x+1), 3-5 the
// walker's row, 6-8 the row below.  Entry: bits 0-1 what the abandon test needs from the empty neighbours walk_rule passed
// over: 0 = the west one (the pixel's west edge is a border edge), 1 = only the east one, 2 = neither; bits 2-4 the s of
// the next step, d ^ 4 for the step direction d; bit 5 set when the step goes up (dir_dy(d) < 0); bits 6-7 dir_dx(d) + 1.
// The step changes row when bits 2-3 are not both zero (d is neither east nor west).
#define STEP_TAB_BYTES 4096
// One table per CTA, in the shared memory of every kernel that calls trace_border (4 KB).  Such a kernel must fill it
// with step_table_build() and synchronise the block before its first trace: the table is not initialised otherwise.
__shared__ uint32_t step_tab[STEP_TAB_BYTES / 4];                // four entries per word, little-endian

// walk_rule's neighbour mask (bit d = neighbour in direction d) of a raw9 neighbourhood
__device__ __forceinline__ uint32_t nbr8_of_raw9(uint32_t r)
{
    return ((r >> 5) & 1u) | (((r >> 2) & 1u) << 1) | (((r >> 1) & 1u) << 2) | ((r & 1u) << 3) |
           (((r >> 3) & 1u) << 4) | (((r >> 6) & 1u) << 5) | (((r >> 7) & 1u) << 6) | (((r >> 8) & 1u) << 7);
}

// Every thread of the block fills its share, the eight entries of a neighbourhood as two words; the block synchronises
// before the first trace reads the table.
__device__ __forceinline__ void step_table_build()
{
    for (int r = threadIdx.x; r < STEP_TAB_BYTES / 8; r += blockDim.x) {
        const uint32_t m = nbr8_of_raw9((uint32_t)r);
        uint32_t w[2] = {0u, 0u};
#pragma unroll
        for (int s = 0; s < 8; ++s) {
            unsigned zeros;
            const int d = walk_rule(m, s, zeros);
            const uint32_t thr = (zeros & (1u << 4)) ? 0u : (zeros & 1u) ? 1u : 2u;
            const uint32_t e = thr | ((uint32_t)(d ^ 4) << 2) | ((dir_dy(d) < 0 ? 1u : 0u) << 5) | ((uint32_t)(dir_dx(d) + 1) << 6);
            w[s >> 2] |= e << (8 * (s & 3));
        }
        step_tab[2 * r] = w[0]; step_tab[2 * r + 1] = w[1];
    }
}

// Step table index (raw9 << 3) + s of column col1 + 1 (-1 <= col1 <= 62) of three 64-bit rows.  At column 0 the triples are
// shifted one bit further, so column -1 reads the zero shifted in.
__device__ __forceinline__ uint32_t step_index(unsigned long long up, unsigned long long mid, unsigned long long dn, int col1, uint32_t s)
{
    const int sh = max(col1, 0);
    const uint32_t k = col1 < 0 ? 4u : 3u;
    const uint32_t u = (uint32_t)(up >> sh) << k, m = (uint32_t)(mid >> sh) << (k + 3), d = (uint32_t)(dn >> sh) << (k + 6);
    return (u & 0x38u) | (m & 0x1c0u) | (d & 0xe00u) | s;
}

template <bool WINDOW> struct GreenAcc { typedef uint32_t T; };
template <> struct GreenAcc<true> { typedef long long T; };

// trace_border's default per-step visitor: none
struct NoVisit { __device__ __forceinline__ void operator()(int, int, int, int) const {} };

// Full trace of the border that starts at the west (side 4) or east (side 0) edge of pixel (x, y) of a box of mw x mh pixels
// (bit rows of wpr words, bits at x >= mw zero).  Writes the Green sums a00/a10/a01 of its CHAIN_APPROX_SIMPLE polygon, the
// perimeter, the number of steps and, given bbox, the bounding box of the border's pixels.  Vertices and edge keys are
// taken in frame coordinates (x + ox, y + oy) of a frame of width Wabs; the frame sizes the library accepts (at most 16384 x
// 16384) keep them in 32 bits.  key0 >= 0: also verify that the start edge, key0 = 2 * (frame pixel index) + east, is the
// border's smallest west/east edge (where cv.findContours starts it); returns 0 as soon as a smaller one is met.  key0 < 0:
// no check.  Returns 1 for a completed trace; *overflow = 1 when the border is longer than WALK_BUDGET steps.
//
// How a step is taken:
//  * the five rows y-2 .. y+2 around the walker live in registers as 64-bit words, and a step looks up its direction in the
//    step table (step_table_build).  When the walker changes row the rows shift and the load of the new outer row is issued
//    at once; it is first read when the walker changes row again, a step later at the soonest (a walker moves one row per
//    step at most), so a step does not wait for a row it requested itself;
//  * the loop body is straight-line code: the Green sums, the bounding box and the abandon and end tests are taken at
//    every step, so the lanes of a warp stay together.  Branches are left for the loop exit, the window slide and the end
//    of a diagonal segment longer than one pixel (rare);
//  * Green sums per unit step instead of per CHAIN_APPROX_SIMPLE vertex: the sums are linear along a straight run, so the
//    terms of a run's unit steps add up exactly to the term of its end points.  Box-local coordinates, translated at the
//    end: a10 = a10' + 3 ox a00, a01 = a01' + 3 oy a00 (exact integer identity for a closed polygon);
//  * bounding box over every pixel of the walk: a pixel of a straight run lies between the run's end vertices;
//  * perimeter: CHAIN_APPROX_SIMPLE segments are the runs of one step direction, axis-parallel (length = an integer, exact in
//    float32) or diagonal (length = float32 sqrt(2 k^2)); the double sum of such float32 values is exact in any order, so
//    axis and diagonal steps are counted, and a longer diagonal is added when its run ends.  The run that closes the border
//    continues the run the trace started on when the start pixel is no vertex.
//
// WINDOW = false: a box at most 64 pixels wide and 1024 high with two words per row, 8-byte aligned; a row is one 64-bit
// load.  In such a box the Green sums stay below 2^29 (|a01'| <= 6 * 2^16 * 2^10), so they are summed modulo 2^32.
// WINDOW = true: any box, e.g. a whole frame (ox = oy = 0, Wabs = mw); rows are read with 32-bit loads only.  The rows are
// seen through a 64-pixel window, first centred on the start pixel, that is re-centred on the walker (five row loads) when
// it reaches a window column whose outer neighbour is not known.  A box at most 64 wide (wpr = 1 or 2) fits the window at
// origin 0, which never moves.  Coordinates then exceed 64, so a10/a01 are summed in 64 bits.
//
// Compile-time extras, off by default:
//  * MIN_KEY: *min_key = the border's smallest west/east edge key 2 * (frame pixel index) + east, the start edge included;
//    a single pixel gives its west edge.  Used with key0 < 0.
//  * visit(x, y, dx, dy) at every step: the walker's pixel in frame coordinates and the step it takes from there.
//
// Precondition: the calling block has filled step_tab (step_table_build) and passed a __syncthreads() since.
template <bool WINDOW, bool MIN_KEY = false, class Visit = NoVisit>
static __device__ int trace_border(const uint32_t* __restrict__ rows, int mh, int wpr, int mw,
                                   int x, int y, int side, long long key0, long long* a, double* per, int* n_chain, int* overflow,
                                   int ox, int oy, int Wabs, int* bbox, long long* min_key = nullptr, Visit visit = Visit())
{
    const int wx0 = WINDOW ? max(min(x - 32, mw - 64), 0) : 0;     // window origin in the box; coordinates below are relative to it
    x -= wx0; ox += wx0;
    int wofs = 0;                                   // window origin relative to wx0 (WINDOW only)
    int wi0 = wx0 >> 5, wsh = wx0 & 31;
    const unsigned long long* rows64 = (const unsigned long long*)rows;                             // rows of a two-word box are 8-byte aligned
    auto load = [&](int yy) -> unsigned long long {
        if ((unsigned)yy >= (unsigned)mh) return 0ull;
        if (!WINDOW) return rows64[(unsigned)yy];
        const uint32_t* r = rows + (size_t)yy * wpr + wi0;         // origin + 63 < mw or origin 0: word wi0 + 1 exists unless wpr = 1
        const uint32_t w0 = r[0], w1 = wpr > 1 ? r[1] : 0u, w2 = (wsh && wi0 + 2 < wpr) ? r[2] : 0u;
        const unsigned long long lo = (unsigned long long)w0 | ((unsigned long long)w1 << 32);
        return wsh ? (lo >> wsh) | ((unsigned long long)w2 << (64 - wsh)) : lo;
    };
    unsigned long long u2 = load(y - 2), up = load(y - 1), mid = load(y), dn = load(y + 1), d2 = load(y + 2);
    if (bbox) { bbox[0] = bbox[2] = x + ox; bbox[1] = bbox[3] = y + oy; }
    // start: clockwise search (side-1, side-2, ... side-7) for the border's predecessor of the start pixel
    uint32_t m0 = nbr8_of_raw9(step_index(up, mid, dn, x - 1, 0) >> 3);
    uint32_t rev = __brev(m0) >> 24, sh = (8 - side) & 7;
    uint32_t r0 = (((rev | (rev << 8)) >> sh) & 0x7fu);           // bit j = m0[(side - 1 - j) & 7], j = 0..6
    if (r0 == 0) {                                              // single pixel
        if (MIN_KEY) *min_key = 2LL * ((long long)(y + oy) * Wabs + x + ox);
        a[0] = a[1] = a[2] = 0; *per = 0.0; *n_chain = 1; return key0 < 0 || side == 4;
    }
    const int s0 = (side - 1 - (__ffs(r0) - 1)) & 7;            // the closing step predecessor -> start goes in direction s0 ^ 4
    const int lin1 = (y + dir_dy(s0)) * Wabs + x + dir_dx(s0);  // the predecessor as cy * Wabs + cx
    // edge keys in 32 bits: key = 2 * (row * Wabs + col) + east = 2 * (oy * Wabs + ox) + 2 * (cy * Wabs + cx) + east.  An edge
    // smaller than key0 is met when kt - 2 * (cy * Wabs + cx) exceeds the step table's threshold (0 for the west edge, 1 for
    // the east edge).
    const int kt = key0 >= 0 ? (int)key0 - 2 * (oy * Wabs + ox) : -(1 << 30);
    int kmin = 2 * (y * Wabs + x) + (side == 0);                // MIN_KEY: smallest edge key so far, relative like kt
    uint32_t a00 = 0;
    typename GreenAcc<WINDOW>::T a10 = 0, a01 = 0;
    int n_diag = 0, n_long = 0;                                 // diagonal steps, those of them on runs longer than one
    double perim_long = 0.0;
    int s = s0, run = -(1 << 30), first_turn = WALK_BUDGET;     // run < 0: no vertex met yet
    int bx0 = x, bx1 = x, by0 = y, by1 = y;
    int wx = x, wy = y;
    int col1 = x - 1;                                           // window column of the walker - 1
    int n = 0;
    bool abandon = false, done = false;
#pragma unroll 1
    while (n < WALK_BUDGET) {
        const uint32_t e = ((const uint8_t*)step_tab)[step_index(up, mid, dn, col1, s)];
        const int sn = (e >> 2) & 7, thr = e & 3;               // sn = d ^ 4 for the step direction d
        const int dx = (int)(e >> 6) - 1, dy = (e & 0x20u) ? -1 : (e & 0x0cu) ? 1 : 0;
        const int lin = wy * Wabs + wx;
        ++n;
        visit(wx + ox, wy + oy, dx, dy);
        if (MIN_KEY && thr < 2) kmin = min(kmin, 2 * lin + thr);
        abandon = thr < 2 && kt - 2 * lin > thr;
        done = lin == lin1 && sn == s0;
        const int dxy = wx * dy - dx * wy;
        a00 += (uint32_t)dxy;
        if (WINDOW) { a10 += (long long)dxy * (2 * wx + dx); a01 += (long long)dxy * (2 * wy + dy); }
        else { a10 += (uint32_t)dxy * (uint32_t)(2 * wx + dx); a01 += (uint32_t)dxy * (uint32_t)(2 * wy + dy); }
        bx0 = min(bx0, wx); bx1 = max(bx1, wx); by0 = min(by0, wy); by1 = max(by1, wy);
        n_diag += sn & 1;
        const bool turn = sn != s;                              // (wx, wy) is a vertex
        if (turn && (s & 1) && run > 1) {                // a diagonal segment longer than one pixel ends here
            perim_long += (double)__fsqrt_rn((float)(2 * run * run));
            n_long += run;
        }
        if (turn) first_turn = min(first_turn, n);
        run = turn ? 1 : run + 1;
        s = sn;
        if (abandon || done) break;
        const int nx = wx + dx, ny = wy + dy;
        col1 += dx;
        bool slide = false;
        if (WINDOW) {
            const int bx = col1 + 1, org = wx0 + wofs;              // window column of the next pixel, window origin in the box
            slide = (bx == 0 && org > 0) || (bx == 63 && org + 64 < mw);
            if (slide) {
                const int norg = min(max(wx0 + nx - 32, 0), mw - 64);
                wofs = norg - wx0; wi0 = norg >> 5; wsh = norg & 31;
                col1 = nx - wofs - 1;
                u2 = load(ny - 2); up = load(ny - 1); mid = load(ny); dn = load(ny + 1); d2 = load(ny + 2);
            }
        }
        if (!slide && dy != 0) {
            const unsigned long long nr = load(ny + 2 * dy);
            if (dy < 0) { d2 = dn; dn = mid; mid = up; up = u2; u2 = nr; }
            else { u2 = up; up = mid; mid = dn; dn = d2; d2 = nr; }
        }
        wx = nx; wy = ny;
    }
    if (MIN_KEY) *min_key = 2LL * ((long long)oy * Wabs + ox) + kmin;
    if (!abandon && !done) {
        *overflow = 1;
        a[0] = a[1] = a[2] = 0; *per = 0.0; *n_chain = n;
        return 0;
    }
    if (abandon) return 0;
    const int k = run + first_turn - 1;                         // the closing segment, in direction s0 ^ 4: the last run and the first
    if ((s0 & 1) && k > 1) { perim_long += (double)__fsqrt_rn((float)(2 * k * k)); n_long += k; }
    const long long A00 = (int)a00;
    a[0] = A00;
    if (WINDOW) { a[1] = a10 + 3LL * ox * A00; a[2] = a01 + 3LL * oy * A00; }
    else { a[1] = (long long)(int)a10 + 3LL * ox * A00; a[2] = (long long)(int)a01 + 3LL * oy * A00; }
    *per = (double)(n - n_diag) + (double)(n_diag - n_long) * (double)__fsqrt_rn(2.0f) + perim_long;
    *n_chain = n;
    if (bbox) { bbox[0] = bx0 + ox; bbox[1] = by0 + oy; bbox[2] = bx1 + ox; bbox[3] = by1 + oy; }
    return 1;
}
