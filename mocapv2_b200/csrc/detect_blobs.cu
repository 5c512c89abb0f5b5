// Blob stage of _find_dot: packed binary image -> 8-connected blobs, contours, centroids.
//
// Replaces lib/ImageOperations.py:41-65 of the reference for a batch of frames:
//     cv.findContours(RETR_TREE, CHAIN_APPROX_SIMPLE) -> contourArea / arcLength filter -> cv.moments centroid
// One CTA per frame, working on the sparse foreground tiles left by filter_tiles:
//   runs        horizontal foreground runs extracted from the 32-bit row words (ffs/popc), bucketed by row
//   labelling   union-find over runs (8-connectivity, smaller raster index wins) -> blob = root run, whose
//               first pixel is the blob's raster-first pixel = start of its outer border (SURVEY App. A5);
//               per-blob pixel sums m00/m10/m01 accumulated with atomics (closed form per run)
//   holes       every run's right edge starts a short Suzuki-Abe walk; the walk that returns to its own
//               start without meeting a smaller west/east edge of the same border is a hole border start
//   contours    one thread per border: border following with CHAIN_APPROX_SIMPLE vertices, Green sums
//               a00/a10/a01 in int64, perimeter = sum of float32 sqrt per segment (exact in double)
//   tree/order  parents from the nearest foreground pixel to the left (Suzuki Table 1), output order =
//               pre-order with siblings in reverse raster order, then the reference's filter and centroid.
#include "common.cuh"
#include "walk.cuh"

#define BLOB_THREADS 256
#define MAX_DEPTH 8
#define RUN_DEAD 0xffffffffu   // run slot emptied by merging (x0 = 0xffff sorts after every live run)

struct BlobWs {                 // per-frame slices of the workspace
    int* rowptr;                // [H + 2]
    int* rowfill;               // [H + 1]
    uint32_t* run_xx;           // [max_runs] x0 | x1 << 16
    uint16_t* run_y;            // [max_runs]
    int* run_parent;            // [max_runs]
    int* run_rank;              // [max_runs] blob rank of a root run (exclusive scan of root flags)
    unsigned long long* run_sum;// [max_runs][3] pixel sums accumulated at the root run
    // contours
    int* c_start;               // [max_contours] start pixel index y*W+x
    int* c_type;                // 0 outer, 1 hole
    int* c_comp;                // blob rank owning the border
    int* c_parent;              // contour index, -1 top level, <= -2: same parent as outer contour (-2 - v)
    long long* c_a;             // [max_contours][3] a00 a10 a01
    double* c_per;              // perimeter
    int* c_n;                   // chain length
    int* c_rank;                // output position
    int* c_keep;
    int* holes_of;              // [max_contours] number of holes per blob
};

__device__ __forceinline__ int uf_find(int* parent, int x)
{
    // path halving: a non-root's parent only ever moves to an ancestor, so the racy plain store is benign
    int p = parent[x];
    while (p != x) {
        int g = parent[p];
        if (g != p) parent[x] = g;
        x = p; p = g;
    }
    return x;
}
__device__ __forceinline__ void uf_union(int* parent, int a, int b)
{
    for (;;) {
        a = uf_find(parent, a);
        b = uf_find(parent, b);
        if (a == b) return;
        if (a < b) { int t = a; a = b; b = t; }       // a > b: hang a under b
        int old = atomicMin(&parent[a], b);
        if (old == a) return;
        a = old;                                      // somebody else re-parented a meanwhile
    }
}

// block-wide exclusive scan helper over an int array in global memory (in place), returns total in *total_s (shared)
__device__ void block_exclusive_scan(int* data, int n, int* sh /*[BLOB_THREADS + 1]*/)
{
    const int tid = threadIdx.x, nt = blockDim.x;
    int chunk = (n + nt - 1) / nt;
    int b = tid * chunk, e = min(b + chunk, n);
    int s = 0;
    for (int k = b; k < e; ++k) s += data[k];
    sh[tid] = s;
    __syncthreads();
    if (tid == 0) {
        int acc = 0;
        for (int k = 0; k < nt; ++k) { int v = sh[k]; sh[k] = acc; acc += v; }
        sh[nt] = acc;
    }
    __syncthreads();
    int acc = sh[tid];
    for (int k = b; k < e; ++k) { int v = data[k]; data[k] = acc; acc += v; }
    __syncthreads();
}

struct BlobParams {
    int H, W, TX;
    int max_fg, max_runs, max_blobs, max_contours;
    double min_area, min_circ;
    int xy_float;                    // centroid records as float32 pairs (sub-pixel), else int32 (store_centroid)
};

__global__ void __launch_bounds__(BLOB_THREADS) blobs_kernel(
    const uint32_t* __restrict__ bits_all, const uint32_t* __restrict__ fg_tiles_all, const int* __restrict__ n_fg_all,
    BlobParams P, char* __restrict__ ws_base, size_t ws_stride,
    int32_t* __restrict__ out_xy, int32_t* __restrict__ out_count, int32_t* __restrict__ out_flags,
    int64_t* __restrict__ out_blob_sums, int32_t* __restrict__ out_blob_count,
    double* __restrict__ out_contours, int32_t* __restrict__ out_contour_count,
    int32_t* __restrict__ out_labels, const int* __restrict__ need_general)
{
    const int f = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    if (need_general && !need_general[f]) return;           // frame fully handled by the cluster path
    const int H = P.H, W = P.W, TX = P.TX;
    __shared__ int sh[BLOB_THREADS + 1];
    __shared__ int s_nblobs, s_nholes, s_flag, s_ncont;

    // carve the per-frame workspace
    char* p = ws_base + (size_t)f * ws_stride;
    BlobWs w;
    auto take = [&](size_t bytes) { char* r = p; p += (bytes + 15) & ~(size_t)15; return r; };
    w.rowptr = (int*)take((size_t)(H + 2) * 4);
    w.rowfill = (int*)take((size_t)(H + 2) * 4);
    w.run_xx = (uint32_t*)take((size_t)P.max_runs * 4);
    w.run_y = (uint16_t*)take((size_t)P.max_runs * 2);
    w.run_parent = (int*)take((size_t)P.max_runs * 4);
    w.run_rank = (int*)take((size_t)(P.max_runs + 1) * 4);
    w.run_sum = (unsigned long long*)take((size_t)P.max_runs * 24);
    w.c_start = (int*)take((size_t)P.max_contours * 4);
    w.c_type = (int*)take((size_t)P.max_contours * 4);
    w.c_comp = (int*)take((size_t)P.max_contours * 4);
    w.c_parent = (int*)take((size_t)P.max_contours * 4);
    w.c_a = (long long*)take((size_t)P.max_contours * 24);
    w.c_per = (double*)take((size_t)P.max_contours * 8);
    w.c_n = (int*)take((size_t)P.max_contours * 4);
    w.c_rank = (int*)take((size_t)P.max_contours * 4);
    w.c_keep = (int*)take((size_t)P.max_contours * 4);
    w.holes_of = (int*)take((size_t)P.max_contours * 4);

    const uint32_t* bits = bits_all + (size_t)f * H * TX;
    const uint32_t* fg_tiles = fg_tiles_all + (size_t)f * P.max_fg;
    BitImg im; im.p = bits; im.W = W; im.H = H; im.WPR = TX;
    int n_t = min(n_fg_all[f], P.max_fg);

    if (tid == 0) { s_flag = 0; s_nholes = 0; }
    for (int y = tid; y < H + 2; y += nt) w.rowptr[y] = 0;
    __syncthreads();

    // ---- runs per row --------------------------------------------------------------------------------------
    for (int it = tid; it < n_t * TILE; it += nt) {
        int t = fg_tiles[it >> 5], r = it & 31;
        int ty = t / TX, tx = t - ty * TX, y = ty * TILE + r;
        if (y >= H) continue;
        uint32_t v = bits[(size_t)y * TX + tx];
        int n = __popc(v & ~(v << 1));
        if (n) atomicAdd(&w.rowptr[y], n);
    }
    __syncthreads();
    block_exclusive_scan(w.rowptr, H + 1, sh);
    const int n_runs = w.rowptr[H];
    if (n_runs > P.max_runs) {
        if (tid == 0) {
            out_flags[f] |= MOCAP_FLAG_RUN_OVERFLOW;
            out_count[f] = 0;
            if (out_blob_count) out_blob_count[f] = 0;
            if (out_contour_count) out_contour_count[f] = 0;
        }
        return;
    }
    for (int y = tid; y < H + 1; y += nt) w.rowfill[y] = w.rowptr[y];
    __syncthreads();
    for (int it = tid; it < n_t * TILE; it += nt) {
        int t = fg_tiles[it >> 5], r = it & 31;
        int ty = t / TX, tx = t - ty * TX, y = ty * TILE + r;
        if (y >= H) continue;
        uint32_t v = bits[(size_t)y * TX + tx];
        int n = __popc(v & ~(v << 1));
        if (!n) continue;
        int slot = atomicAdd(&w.rowfill[y], n);
        while (v) {
            int a = __ffs(v) - 1;
            uint32_t sh_v = v >> a;
            int len = (sh_v == 0xffffffffu) ? 32 : (__ffs(~sh_v) - 1);
            uint32_t mask = (len >= 32) ? 0xffffffffu : (((1u << len) - 1u) << a);
            v &= ~mask;
            int x0 = tx * TILE + a, x1 = x0 + len - 1;
            w.run_xx[slot] = (uint32_t)x0 | ((uint32_t)x1 << 16);
            w.run_y[slot] = (uint16_t)y;
            ++slot;
        }
    }
    __syncthreads();
    // sort the (few) runs of every row by x0 and merge runs split at a 32-bit word boundary; the slots freed by
    // merging become DEAD runs parked at the end of the row (rowfill[y] = end of the row's live runs)
    for (int y = tid; y < H; y += nt) {
        int b = w.rowptr[y], e = w.rowptr[y + 1];
        for (int i = b + 1; i < e; ++i) {
            uint32_t v = w.run_xx[i];
            int k = i - 1;
            while (k >= b && (w.run_xx[k] & 0xffff) > (v & 0xffff)) { w.run_xx[k + 1] = w.run_xx[k]; --k; }
            w.run_xx[k + 1] = v;
        }
        int wpos = b;
        for (int i = b; i < e; ++i) {
            uint32_t v = w.run_xx[i];
            if (wpos > b && (w.run_xx[wpos - 1] >> 16) + 1 == (v & 0xffff)) w.run_xx[wpos - 1] = (w.run_xx[wpos - 1] & 0xffff) | (v & 0xffff0000u);
            else w.run_xx[wpos++] = v;
        }
        for (int i = wpos; i < e; ++i) w.run_xx[i] = RUN_DEAD;
        w.rowfill[y] = wpos;
    }
    __syncthreads();

    int n_blobs = 0, n_cont = 0, n_arr = 0;        // n_arr: extent of the contour arrays (fast path keeps rejected candidates)
    bool fast_done = false;
    const bool need_labels = out_labels != nullptr || out_blob_sums != nullptr || out_blob_count != nullptr;

    // ---- fast path (no label outputs wanted): border starts straight from the runs --------------------------------------
    // An outer border starts at the first pixel of a run with no 8-neighbour in the row above (necessary condition); a
    // hole border at the last pixel of a run whose gap to the next run is completely covered by one run of the row above.
    // Every candidate is traced once; the trace is discarded as soon as it meets a smaller west/east edge of its border
    // (then it is not where cv.findContours starts that border).  Frames with a hole border fall through to the general
    // path, which needs the labels for the contour tree.
    if (!need_labels) {
        if (tid == 0) { s_ncont = 0; s_nholes = 0; }
        __syncthreads();
        for (int r = tid; r < n_runs; r += nt) {
            uint32_t xx = w.run_xx[r];
            if (xx == RUN_DEAD) continue;
            int y = w.run_y[r], x0 = xx & 0xffff, x1 = xx >> 16;
            int nx0 = (r + 1 < w.rowfill[y]) ? (int)(w.run_xx[r + 1] & 0xffff) : -1;
            bool top = true, covered = false;
            if (y > 0) {
                int lim = nx0 >= 0 ? nx0 : x1 + 1;
                for (int k = w.rowptr[y - 1]; k < w.rowfill[y - 1]; ++k) {
                    uint32_t kk = w.run_xx[k];
                    int k0 = kk & 0xffff, k1 = kk >> 16;
                    if (k0 > lim) break;
                    if (k1 >= x0 - 1 && k0 <= x1 + 1) top = false;
                    if (nx0 >= 0 && k0 <= x1 + 1 && k1 >= nx0 - 1) covered = true;
                }
            }
            if (top) {
                int k = atomicAdd(&s_ncont, 1);
                if (k < P.max_contours) { w.c_start[k] = y * W + x0; w.c_type[k] = 0; }
            }
            if (covered) {
                int k = atomicAdd(&s_ncont, 1);
                if (k < P.max_contours) { w.c_start[k] = y * W + x1; w.c_type[k] = 1; }
            }
        }
        __syncthreads();
        const int n_cand = s_ncont;
        __syncthreads();
        if (n_cand <= P.max_contours) {
            for (int c = tid; c < n_cand; c += nt) {
                int st = w.c_start[c], ty = w.c_type[c], ovf = 0;
                int ok = trace_contour(im, st % W, st / W, ty ? 0 : 4, 2LL * st + ty, &w.c_a[3 * c], &w.c_per[c], &w.c_n[c], &ovf, 0, 0, W);
                if (ovf) atomicOr(&s_flag, MOCAP_FLAG_TRACE_OVERFLOW);
                w.c_keep[c] = ok;                      // parked: candidate is a real border start
                if (ok && ty) atomicAdd(&s_nholes, 1);
            }
            __syncthreads();
            if (s_nholes == 0 && !(s_flag & MOCAP_FLAG_TRACE_OVERFLOW)) {
                // only top-level outer borders: output order = reverse raster order of the start pixels
                for (int c = tid; c < n_cand; c += nt) {
                    int rank = -1;
                    if (w.c_keep[c]) {
                        rank = 0;
                        int st = w.c_start[c];
                        for (int u = 0; u < n_cand; ++u) rank += (w.c_keep[u] && w.c_start[u] > st);
                    }
                    w.c_rank[c] = rank;
                    w.c_parent[c] = -1;
                }
                if (tid == 0) { int nb = 0; for (int c = 0; c < n_cand; ++c) nb += w.c_keep[c] != 0; s_nblobs = nb; }
                __syncthreads();
                n_blobs = s_nblobs; n_cont = n_blobs; n_arr = n_cand;
                fast_done = true;
            }
        }
        if (!fast_done) {
            __syncthreads();
            if (tid == 0) { s_nholes = 0; s_flag &= ~MOCAP_FLAG_TRACE_OVERFLOW; }
            __syncthreads();
        }
    }

    if (!fast_done) {
    // ---- general path: labelling by union-find over runs (8-connectivity) ------------------------------------------------
    for (int r = tid; r < n_runs; r += nt) {
        w.run_parent[r] = r;
        w.run_sum[3 * r] = 0; w.run_sum[3 * r + 1] = 0; w.run_sum[3 * r + 2] = 0;
    }
    __syncthreads();
    for (int r = tid; r < n_runs; r += nt) {
        uint32_t xx = w.run_xx[r];
        if (xx == RUN_DEAD) continue;
        int y = w.run_y[r];
        int x0 = xx & 0xffff, x1 = xx >> 16;
        if (y > 0) {
            for (int k = w.rowptr[y - 1]; k < w.rowfill[y - 1]; ++k) {
                uint32_t kk = w.run_xx[k];
                int k0 = kk & 0xffff, k1 = kk >> 16;
                if (k0 > x1 + 1) break;
                if (k1 >= x0 - 1) uf_union(w.run_parent, r, k);
            }
        }
    }
    __syncthreads();
    for (int r = tid; r < n_runs; r += nt) {
        int root = uf_find(w.run_parent, r);
        w.run_parent[r] = root;          // races only write the same final value or an ancestor -> still valid
    }
    __syncthreads();
    for (int r = tid; r < n_runs; r += nt) {
        uint32_t xx = w.run_xx[r];
        bool live = xx != RUN_DEAD;
        int root = uf_find(w.run_parent, r);
        w.run_parent[r] = root;
        if (live) {
            unsigned long long x0 = xx & 0xffff, x1 = xx >> 16, len = x1 - x0 + 1, y = w.run_y[r];
            atomicAdd(&w.run_sum[3 * root], len);
            atomicAdd(&w.run_sum[3 * root + 1], (x0 + x1) * len / 2);
            atomicAdd(&w.run_sum[3 * root + 2], y * len);
        }
        w.run_rank[r] = (live && root == r) ? 1 : 0;
    }
    if (tid == 0) w.run_rank[n_runs] = 0;
    __syncthreads();
    block_exclusive_scan(w.run_rank, n_runs + 1, sh);
    n_blobs = w.run_rank[n_runs];
    if (out_blob_count && tid == 0) out_blob_count[f] = n_blobs;
    if (n_blobs > P.max_contours) {
        if (tid == 0) {
            out_flags[f] |= MOCAP_FLAG_CONTOUR_OVERFLOW;
            out_count[f] = 0;
            if (out_contour_count) out_contour_count[f] = 0;
        }
        return;
    }
    // blob records + outer contours (index = blob rank)
    for (int r = tid; r < n_runs; r += nt) {
        if (w.run_xx[r] == RUN_DEAD || w.run_parent[r] != r) continue;
        int k = w.run_rank[r];
        if (out_blob_sums && k < P.max_blobs)
            for (int q = 0; q < 3; ++q) out_blob_sums[((size_t)f * P.max_blobs + k) * 3 + q] = (int64_t)w.run_sum[3 * r + q];
        w.c_start[k] = (int)w.run_y[r] * W + (int)(w.run_xx[r] & 0xffff);
        w.c_type[k] = 0;
        w.c_comp[k] = k;
        w.holes_of[k] = 0;
    }
    if (out_labels) {
        int32_t* lab = out_labels + (size_t)f * H * W;
        for (int r = tid; r < n_runs; r += nt) {
            uint32_t xx = w.run_xx[r];
            if (xx == RUN_DEAD) continue;
            int k = w.run_rank[w.run_parent[r]] + 1;
            int y = w.run_y[r];
            for (int x = xx & 0xffff; x <= (int)(xx >> 16); ++x) lab[(size_t)y * W + x] = k;
        }
    }
    __syncthreads();

    // ---- hole borders: canonical east edges ---------------------------------------------------------------------
    for (int r = tid; r < n_runs; r += nt) {
        uint32_t xx = w.run_xx[r];
        if (xx == RUN_DEAD) continue;
        int y = w.run_y[r];
        int x1 = xx >> 16;
        int ovf = 0;
        if (walk_min_edge(im, x1, y, 0, 0, nullptr, &ovf)) {
            int k = n_blobs + atomicAdd(&s_nholes, 1);
            if (k < P.max_contours) {
                int comp = w.run_rank[w.run_parent[r]];
                w.c_start[k] = y * W + x1;
                w.c_type[k] = 1;
                w.c_comp[k] = comp;
                atomicAdd(&w.holes_of[comp], 1);
            }
        }
        if (ovf) atomicOr(&s_flag, MOCAP_FLAG_TRACE_OVERFLOW);
    }
    __syncthreads();
    n_cont = n_blobs + s_nholes;
    n_arr = n_cont;
    if (n_cont > P.max_contours || (s_flag & MOCAP_FLAG_TRACE_OVERFLOW)) {
        if (tid == 0) {
            out_flags[f] |= (n_cont > P.max_contours ? MOCAP_FLAG_CONTOUR_OVERFLOW : 0) | s_flag;
            out_count[f] = 0;
            if (out_contour_count) out_contour_count[f] = 0;
        }
        return;
    }

    // ---- trace every border -------------------------------------------------------------------------------------
    for (int c = tid; c < n_cont; c += nt) {
        int st = w.c_start[c];
        int ovf = 0;
        trace_contour(im, st % W, st / W, w.c_type[c] ? 0 : 4, -1, &w.c_a[3 * c], &w.c_per[c], &w.c_n[c], &ovf, 0, 0, W);
        if (ovf) atomicOr(&s_flag, MOCAP_FLAG_TRACE_OVERFLOW);
    }
    // ---- parents ------------------------------------------------------------------------------------------------
    for (int c = tid; c < n_cont; c += nt) {
        if (w.c_type[c]) { w.c_parent[c] = w.c_comp[c]; continue; }
        // outer border: nearest foreground pixel to the left of the blob's first pixel, on the same row
        int st = w.c_start[c], y = st / W, x0 = st - y * W;
        // locate the root run: binary search not needed, rows hold few runs
        int b = w.rowptr[y], e = w.rowfill[y], r = b;
        while (r < e && (int)(w.run_xx[r] & 0xffff) != x0) ++r;
        if (r == b) { w.c_parent[c] = -1; continue; }
        int q = r - 1;                                    // run ending left of us
        int other = w.run_rank[w.run_parent[q]];          // blob owning it
        if (w.holes_of[other] == 0) { w.c_parent[c] = -2 - other; continue; }
        long long mk; int ovf = 0;
        walk_min_edge(im, (int)(w.run_xx[q] >> 16), y, 0, 1, &mk, &ovf);
        if (ovf) atomicOr(&s_flag, MOCAP_FLAG_TRACE_OVERFLOW);
        if ((mk & 1) == 0) { w.c_parent[c] = -2 - other; continue; }     // smallest edge is a west edge: outer border of `other`
        int hole_start = (int)(mk >> 1), par = -1;
        for (int h = n_blobs; h < n_cont; ++h) if (w.c_start[h] == hole_start) { par = h; break; }
        w.c_parent[c] = par;
    }
    __syncthreads();
    for (int c = tid; c < n_blobs; c += nt) {             // resolve "same parent as the blob on my left"
        int v = w.c_parent[c], guard = 0;
        while (v <= -2 && guard++ < n_blobs) v = w.c_parent[-2 - v];
        w.c_rank[c] = v;                                  // park the resolved parent
    }
    __syncthreads();
    for (int c = tid; c < n_blobs; c += nt) w.c_parent[c] = w.c_rank[c];
    __syncthreads();

    // ---- output order: pre-order, siblings by descending start pixel ------------------------------------------------
    // ancestor chain of start keys, root first; u precedes v iff at the first difference u's key is larger,
    // or u's chain is a proper prefix of v's.
    bool deep = false;
    for (int c = tid; c < n_cont; c += nt) {
        int chain_c[MAX_DEPTH], dc = 0;
        for (int v = c; v >= 0; v = w.c_parent[v]) { if (dc == MAX_DEPTH) { deep = true; break; } chain_c[dc++] = w.c_start[v]; }
        int before = 0;
        for (int u = 0; u < n_cont && !deep; ++u) {
            if (u == c) continue;
            int chain_u[MAX_DEPTH], du = 0;
            for (int v = u; v >= 0; v = w.c_parent[v]) { if (du == MAX_DEPTH) { deep = true; break; } chain_u[du++] = w.c_start[v]; }
            if (deep) break;
            // compare from the root end
            int iu = du - 1, ic = dc - 1, res = 0;    // res: 1 = u first, -1 = c first
            while (iu >= 0 && ic >= 0) {
                if (chain_u[iu] != chain_c[ic]) { res = chain_u[iu] > chain_c[ic] ? 1 : -1; break; }
                --iu; --ic;
            }
            if (res == 0) res = (iu < 0) ? 1 : -1;    // the shorter chain is the ancestor
            before += res > 0;
        }
        w.c_rank[c] = before;
    }
    if (deep) atomicOr(&s_flag, MOCAP_FLAG_DEPTH_OVERFLOW);
    __syncthreads();
    if (s_flag & MOCAP_FLAG_DEPTH_OVERFLOW) {
        // slow, fully general path: one thread walks the tree
        if (tid == 0) {
            int pos = 0, cur = -1;                 // cur = node whose children we enumerate; -1 = top level
            // iterative DFS without a stack: c_keep temporarily stores "largest child key already emitted"
            for (int c = 0; c < n_cont; ++c) w.c_keep[c] = 0x7fffffff;
            int top_limit = 0x7fffffff;
            while (true) {
                int limit = cur < 0 ? top_limit : w.c_keep[cur];
                int best = -1;
                for (int c = 0; c < n_cont; ++c)
                    if (w.c_parent[c] == cur && w.c_start[c] < limit && (best < 0 || w.c_start[c] > w.c_start[best])) best = c;
                if (best >= 0) {
                    if (cur < 0) top_limit = w.c_start[best]; else w.c_keep[cur] = w.c_start[best];
                    w.c_rank[best] = pos++;
                    cur = best;
                } else {
                    if (cur < 0) break;
                    cur = w.c_parent[cur];
                }
            }
        }
        __syncthreads();
    }
    }   // general path

    // ---- the reference's filter and centroid (ImageOperations.py:43-65) -------------------------------------------------
    for (int c = tid; c < n_arr; c += nt) {
        if (w.c_rank[c] < 0) { w.c_keep[c] = 0; continue; }     // rejected fast-path candidate
        long long a00 = w.c_a[3 * c];
        double area = (double)(a00 < 0 ? -a00 : a00) * 0.5;
        double per = w.c_per[c];
        int keep = 0;
        if (per != 0.0) {
            double circ = __ddiv_rn(__dmul_rn(12.566370614359172, area), __dmul_rn(per, per));
            keep = (circ > P.min_circ && area > P.min_area) ? 1 : 0;
        }
        if (a00 == 0) keep = 0;                          // moments["m00"] == 0 -> no centroid
        w.c_keep[c] = keep;
    }
    __syncthreads();
    if (tid == 0) s_ncont = 0;
    __syncthreads();
    for (int c = tid; c < n_arr; c += nt) {
        int rank = w.c_rank[c];
        if (rank < 0) continue;
        long long a00 = w.c_a[3 * c], a10 = w.c_a[3 * c + 1], a01 = w.c_a[3 * c + 2];
        if (out_contours && rank < P.max_contours) {
            double* o = out_contours + ((size_t)f * P.max_contours + rank) * 8;
            int par = w.c_parent[c];
            o[0] = (double)a00; o[1] = (double)a10; o[2] = (double)a01; o[3] = w.c_per[c];
            o[4] = (double)w.c_type[c]; o[5] = (double)(par >= 0 ? w.c_rank[par] : -1);
            o[6] = (double)w.c_keep[c]; o[7] = (double)w.c_start[c];
        }
        if (!w.c_keep[c]) continue;
        int pos = 0;
        for (int u = 0; u < n_arr; ++u) pos += (w.c_keep[u] && w.c_rank[u] < rank);
        atomicAdd(&s_ncont, 1);
        if (pos < P.max_blobs) {
            double sgn = a00 > 0 ? 1.0 : -1.0;
            double m00 = __dmul_rn((double)a00, sgn * 0.5);
            double m10 = __dmul_rn((double)a10, sgn * 0.16666666666666666);
            double m01 = __dmul_rn((double)a01, sgn * 0.16666666666666666);
            store_centroid(out_xy + ((size_t)f * P.max_blobs + pos) * 2, __ddiv_rn(m10, m00), __ddiv_rn(m01, m00), P.xy_float);
        }
    }
    __syncthreads();
    if (tid == 0) {
        int kept = s_ncont;
        int fl = s_flag;
        if (kept > P.max_blobs) { fl |= MOCAP_FLAG_BLOB_OVERFLOW; kept = P.max_blobs; }
        out_count[f] = kept;
        out_flags[f] |= fl | (need_general ? (MOCAP_FLAG_GENERAL_PATH | (need_general[f] << 8)) : 0);   // bits 8.. = why (informational)
        if (out_contour_count) out_contour_count[f] = n_cont;
    }
}

// foreground-tile list of a dense packed binary image (stage entry mocap_blobs_batch; the fused path gets it from filter_tiles)
__global__ void tiles_from_bits_kernel(const uint32_t* __restrict__ bits, int n, int H, int TX, int TY,
                                       uint32_t* __restrict__ fg_tiles, int* __restrict__ n_fg, int max_fg)
{
    long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)n * TX * TY) return;
    int f = (int)(idx / (TX * TY)), t = (int)(idx - (long long)f * TX * TY);
    int ty = t / TX, tx = t - ty * TX;
    uint32_t any = 0;
    for (int r = 0; r < TILE && ty * TILE + r < H; ++r) any |= bits[((size_t)f * H + ty * TILE + r) * TX + tx];
    if (any) {
        int slot = atomicAdd(&n_fg[f], 1);
        if (slot < max_fg) fg_tiles[(size_t)f * max_fg + slot] = (uint32_t)t;
    }
}

int launch_tiles_from_bits(const uint32_t* bits, int n, int H, int TX, int TY, uint32_t* fg_tiles, int* n_fg, int max_fg, cudaStream_t s)
{
    CUDA_TRY(cudaMemsetAsync(n_fg, 0, (size_t)n * sizeof(int), s));
    long long total = (long long)n * TX * TY;
    LAUNCH(tiles_from_bits_kernel, (unsigned)((total + 255) / 256), 256, 0, s, bits, n, H, TX, TY, fg_tiles, n_fg, max_fg);
    CUDA_TRY(cudaGetLastError());
    return MOCAP_OK;
}

size_t blob_ws_stride(int H, int max_runs, int max_contours)
{
    size_t b = 0;
    auto add = [&](size_t bytes) { b += (bytes + 15) & ~(size_t)15; };
    add((size_t)(H + 2) * 4); add((size_t)(H + 2) * 4);
    add((size_t)max_runs * 4); add((size_t)max_runs * 2); add((size_t)max_runs * 4); add((size_t)(max_runs + 1) * 4);
    add((size_t)max_runs * 24);
    for (int k = 0; k < 4; ++k) add((size_t)max_contours * 4);
    add((size_t)max_contours * 24); add((size_t)max_contours * 8);
    for (int k = 0; k < 4; ++k) add((size_t)max_contours * 4);
    return (b + 255) & ~(size_t)255;
}

int launch_blobs(const uint32_t* bits, const uint32_t* fg_tiles, const int* n_fg, int n, int H, int W, int TX,
                 int max_fg, int max_runs, int max_blobs, int max_contours, double min_area, double min_circ,
                 char* ws, size_t ws_stride,
                 int32_t* out_xy, int xy_float, int32_t* out_count, int32_t* out_flags,
                 int64_t* out_blob_sums, int32_t* out_blob_count, double* out_contours, int32_t* out_contour_count,
                 int32_t* out_labels, const int* need_general, cudaStream_t s)
{
    BlobParams P;
    P.H = H; P.W = W; P.TX = TX; P.max_fg = max_fg; P.max_runs = max_runs; P.max_blobs = max_blobs;
    P.max_contours = max_contours; P.min_area = min_area; P.min_circ = min_circ; P.xy_float = xy_float;
    LAUNCH(blobs_kernel, n, BLOB_THREADS, 0, s, bits, fg_tiles, n_fg, P, ws, ws_stride, out_xy, out_count, out_flags,
                                            out_blob_sums, out_blob_count, out_contours, out_contour_count, out_labels, need_general);
    CUDA_TRY(cudaGetLastError());
    return MOCAP_OK;
}


// ---------------------------------------------------------------------------------------------------------
// cv.drawContours(img, contours_filtered, -1, (0, 0, 255), 2) of _find_dot (lib/ImageOperations.py:52-55), display only: on the
// one-channel image the colour is its first component, 0.  A thickness-2 polyline through the CHAIN_APPROX_SIMPLE vertices of a
// border (OpenCV widens every segment by one pixel to each side and rounds its ends with a radius-1 disc) covers exactly: the plus-
// shaped neighbourhood of every border pixel and, for every diagonal step (x, y) -> (x + dx, y + dy), the pixels (x + dx, y),
// (x, y + dy), (x + dx, y - dy), (x - dx, y + dy), (x + 2 dx, y), (x, y + 2 dy) (checked against cv2 on random images with holes and
// nesting, tests/test_dropin.py).  One thread per kept contour of the table re-walks its border on the packed binary image.
// ---------------------------------------------------------------------------------------------------------
__global__ void draw_contours_kernel(const uint32_t* __restrict__ bits, const double* __restrict__ contours, const int32_t* __restrict__ contour_count,
                                     int max_contours, int H, int W, int TX, uint8_t* __restrict__ img, int value)
{
    const int f = blockIdx.y, c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= min(contour_count[f], max_contours)) return;
    const double* o = contours + ((size_t)f * max_contours + c) * 8;
    if (o[6] == 0.0) return;                                   // not kept by the area / circularity filter
    const int st = (int)o[7], hole = o[4] != 0.0;
    BitImg im; im.p = bits + (size_t)f * H * TX; im.W = W; im.H = H; im.WPR = TX;
    uint8_t* out = img + (size_t)f * H * W;
    auto put = [&](int x, int y) { if ((unsigned)x < (unsigned)W && (unsigned)y < (unsigned)H) out[(size_t)y * W + x] = (uint8_t)value; };
    auto plus = [&](int x, int y) { put(x, y); put(x - 1, y); put(x + 1, y); put(x, y - 1); put(x, y + 1); };
    const int y0 = st / W, x0 = st - y0 * W;
    Walk w; walk_init(im, w, x0, y0, hole ? 0 : 4);           // outer borders start on a west edge, hole borders on an east edge
    plus(x0, y0);
    if (w.single) return;
    for (int step = 0; step < WALK_BUDGET; ++step) {
        const int cx = w.x, cy = w.y;
        unsigned zeros; bool done;
        const int d = walk_step(im, w, zeros, done);
        plus(cx, cy);
        if (d & 1) {
            const int dx = dir_dx(d), dy = dir_dy(d);
            put(cx + dx, cy); put(cx, cy + dy); put(cx + dx, cy - dy); put(cx - dx, cy + dy); put(cx + 2 * dx, cy); put(cx, cy + 2 * dy);
        }
        if (done) break;
    }
}

extern "C" int mocap_draw_contours_batch(const uint32_t* bits_dev, const double* contours_dev, const int32_t* contour_count_dev,
                                         int n_frames, int H, int W, int max_contours, uint8_t* img_dev, int value, void* stream)
{
    if (!bits_dev || !contours_dev || !contour_count_dev || !img_dev || n_frames <= 0 || n_frames > 65535 || H <= 0 || W <= 0 || max_contours <= 0)
        return MOCAP_ERR_INVALID;
    LAUNCH(draw_contours_kernel, dim3(cdiv(max_contours, 64), n_frames), 64, 0, (cudaStream_t)stream, bits_dev, contours_dev, contour_count_dev,
           max_contours, H, W, cdiv(W, TILE), img_dev, value);
    CUDA_TRY(cudaGetLastError());
    return MOCAP_OK;
}
