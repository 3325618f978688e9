// kernels_tracker.cu — K11 + K12: the nubotracker per-frame path, gstnubotracker.cpp:356-377, as ONE fused kernel:
//   cvtColor(BGRA->gray) :356, absdiff(gray, img_prev) :361, threshold(diff, thr, 255, BINARY) :364,
//   updateMotionHistory(mask, mhi, ts, MHI_DURATION=0.2) :368, segmentMotion(mhi, ts, 32) :376,
//   img_prev = gray :419.  calcMotionGradient (:372) writes two outputs nobody reads and is skipped.
//
// segmentMotion is connected-component labelling: 4-connected pixels are joined when their MHI values differ by at
// most 32 (OpenCV's floating-range flood fill with lo = up = segThresh), zeros never join anything that matters
// (OpenCV swaps them for FLT_MAX*0.1), a component is reported iff it contains a pixel with mhi == ts, in raster order
// of its first such pixel, with the bounding box of ALL its pixels.
//
// Layout.  The motion history holds, per pixel, either 0 or the (float) timestamp of one earlier frame, so it is stored
// as ONE BYTE per pixel: an index into a per-context table of the live timestamps (host side, context.cu: an entry is
// live while value >= ts - duration; equal float values share an index; 255 live values at most — the reference's
// 0.2 ms duration keeps one).  Per frame and pixel the kernel reads 4 (BGRA) + 1 (prev) + 1 (history) bytes and writes
// 1 + 1: 8 bytes, against 38 in the round-1 kernels (float history, an int label, an int seed and an int4 box per pixel).
//
// One 64 x 16 tile per 256-thread block (64 x 32 with -DTRK_TH=32: the round-2 default until its last session — the smaller
// tile halves the slowest block and is 2-3 us faster at every frame size), four pixels per thread (128-bit BGRA loads):
//   1. point operations, the new history values of the tile land in shared memory;
//   2. block-local labelling in shared memory: horizontal pre-linking inside each thread's four pixels, then lock-free
//      union-find (atomicMin links, the smaller index wins, so a root is its component's first pixel in raster order);
//   3. per-root bounding box / first-seed reductions: per run of equal roots inside a thread's four pixels, then per warp
//      (one REDUX when the warp sees a single component, which is the case inside a blob), then shared-memory atomics;
//   4. components that stay inside the tile are final: reported at once.  Components on the tile's perimeter go to a
//      small per-tile table (<= 192 slots), and the tile publishes the slot of each perimeter pixel;
//   5. each tile edge is stitched by whichever of its two tiles arrives second (an arrival counter per edge): union-find
//      over the slots, across tiles, in global memory;
//   6. the last block to finish folds the slot records into their roots, appends those that own a seed, and writes the
//      components in raster order of their first seed.  Counters and edge flags are re-armed on the way: the kernel cleans
//      up after itself.
// No second launch, no grid-wide barrier: nothing ever waits for another block.
#include <limits.h>

#include "internal.h"

#define TRK_MAX_COMPONENTS 16384
#define TRK_TW 64
#ifndef TRK_TH
#define TRK_TH 16                                    // 16 or 32: rows of a tile (a thread owns one unit of four pixels per 16 rows)
#endif
#define TRK_NH (TRK_TH / 16)
#define TRK_NPX (TRK_TW * TRK_TH)
#define TRK_PERIM (2 * TRK_TW + 2 * TRK_TH)          // top 0..63, bottom 64..127, then the left and the right column
#define TRK_SLOTS TRK_PERIM
#define TRK_NONE 0x7fffffff

// -DNV_TRK_TRACE: clock64 at a dozen checkpoints of every block (tools/trk_trace.py builds that variant and prints the phases)
#ifdef NV_TRK_TRACE
__device__ long long g_trk_trace[4096 * 16];
#define TRK_T(k) do { if (threadIdx.x == 0 && blockIdx.x < 4096) g_trk_trace[blockIdx.x * 16 + (k)] = clock64(); } while (0)
extern "C" __attribute__((visibility("default"))) int nv_debug_trk_trace(long long *out, int nblocks)
{
    return (int)cudaMemcpyFromSymbol(out, g_trk_trace, sizeof(long long) * 16 * (size_t)(nblocks < 4096 ? nblocks : 4096));
}
#else
#define TRK_T(k) do { } while (0)
#endif

struct TrkParams {
    SrcPlanes src;
    int w, h, first, thr, cur, ntx, nty, vec;
    uint8_t *prev, *hist;
    unsigned short *bslot;          // [ntiles][TRK_PERIM]: slot of each perimeter pixel, 0xffff = no history there
    int *bcount;                    // [ntiles]
    int4 *bbox;                     // [ntiles][TRK_SLOTS]: min x, min y, max x, max y (image coordinates)
    int *bseed;                     // [ntiles][TRK_SLOTS]: first seed pixel (y * w + x) or TRK_NONE
    int *parent;                    // [ntiles * TRK_SLOTS]
    int *slotlist;                  // [ntiles * TRK_SLOTS]: every used slot (tile * TRK_SLOTS + s), appended tile by tile
    int *edge_flag;                 // arrival counters, one per tile edge
    int *counters;                  // [0] components appended, [1] blocks done, [2] slots in use (all tiles)
    int *keys;                      // [TRK_MAX_COMPONENTS]
    int4 *rects;                    // [TRK_MAX_COMPONENTS]
    int4 *out;                      // [1 + TRK_MAX_COMPONENTS]: (count, 0, 0, 0), rects in raster order of the first seed
    int4 *hout;                     // the context's page-locked copy of out[0 .. 1024] (mapped host memory): written by the last block,
                                    // so that no device-to-host copy follows the launch
    float val[256];                 // timestamp of history index k after this frame's expiry (0: none / expired)
};

__device__ __forceinline__ bool trk_joined(float a, float b)
{
    float d = b - a;
    return a != 0.f && b != 0.f && d >= -32.f && d <= 32.f;       // SEGMENTATION, gstnubotracker.cpp:31
}

template <typename T>
__device__ __forceinline__ int trk_find(T *L, int a)
{
    int p;
    while ((p = ((volatile int *)L)[a]) != a) a = p;
    return a;
}

__device__ __forceinline__ void trk_union(int *L, int a, int b)
{
    bool done;
    do {
        a = trk_find(L, a);
        b = trk_find(L, b);
        if (a < b) { int old = atomicMin(&L[b], a); done = old == b; b = old; }
        else if (b < a) { int old = atomicMin(&L[a], b); done = old == a; a = old; }
        else done = true;
    } while (!done);
}

__device__ __forceinline__ int trk_gray(int b, int g, int r) { return (b * 3735 + g * 19235 + r * 9798 + 16384) >> 15; }

// perimeter position k of a tile -> local pixel index
__device__ __forceinline__ int trk_perim_px(int k)
{
    if (k < TRK_TW) return k;
    if (k < 2 * TRK_TW) return (TRK_TH - 1) * TRK_TW + (k - TRK_TW);
    if (k < 2 * TRK_TW + TRK_TH) return (k - 2 * TRK_TW) * TRK_TW;
    return (k - 2 * TRK_TW - TRK_TH) * TRK_TW + TRK_TW - 1;
}

// stitches the edge between tile a (left / upper) and tile b (right / lower); vertical != 0: b lies below a.  Runs on the
// first two warps of the block (an edge is at most 64 pixels long); a pixel pair that repeats its left neighbour's
// (slot, slot) pair is skipped: along a blob that leaves one union per edge instead of one per pixel.
__device__ void trk_stitch(const TrkParams &P, const float *s_val, int a, int b, int vertical)
{
    if (threadIdx.x >= 64) return;
    const int ax0 = (a % P.ntx) * TRK_TW, ay0 = (a / P.ntx) * TRK_TH, bx0 = (b % P.ntx) * TRK_TW, by0 = (b / P.ntx) * TRK_TH;
    const int len = vertical ? TRK_TW : TRK_TH, i = threadIdx.x, lane = threadIdx.x & 31;
    int xa, ya, xb, yb, ka, kb;
    if (vertical) { xa = ax0 + i; ya = ay0 + TRK_TH - 1; xb = bx0 + i; yb = by0; ka = TRK_TW + i; kb = i; }
    else { xa = ax0 + TRK_TW - 1; ya = ay0 + i; xb = bx0; yb = by0 + i; ka = 2 * TRK_TW + TRK_TH + i; kb = 2 * TRK_TW + i; }
    unsigned sa = 0xffffu, sb = 0xffffu;
    bool joined = false;
    if (i < len && xa < P.w && xb < P.w && ya < P.h && yb < P.h) {
        sa = __ldcg(P.bslot + (size_t)a * TRK_PERIM + ka); sb = __ldcg(P.bslot + (size_t)b * TRK_PERIM + kb);
        if (sa != 0xffffu && sb != 0xffffu)
            joined = trk_joined(s_val[__ldcg(P.hist + (size_t)ya * P.w + xa)], s_val[__ldcg(P.hist + (size_t)yb * P.w + xb)]);
    }
    const unsigned key = joined ? (sa << 16) | sb : 0xffffffffu, left = __shfl_up_sync(0xffffffffu, key, 1);
    if (joined && (lane == 0 || left != key)) trk_union(P.parent, a * TRK_SLOTS + (int)sa, b * TRK_SLOTS + (int)sb);
}

// FMT 0: BGRA (the reference's caps, gstnubotracker.cpp:57-61); 1 / 2 / 3: I420 / NV12 / NV21 planes — the 4:2:0 ingest
// extension: gray = BGR2GRAY(cvtColor(COLOR_YUV2BGR_*)) per pixel, the BGRA frame is never built.
template <int FMT>
__global__ void __launch_bounds__(256) k_trk_fused(const __grid_constant__ TrkParams P)
{
    __shared__ float s_val[256];
    __shared__ union { float m[TRK_NPX]; int minx[TRK_NPX]; } s_a;          // history values, then (labels final) min x per root
    __shared__ int s_lab[TRK_NPX], s_maxx[TRK_NPX], s_maxy[TRK_NPX], s_seed[TRK_NPX];
    __shared__ int s_nslots, s_edges[4], s_last, s_base;

    const int tid = threadIdx.x, lane = tid & 31;
    const int tile = blockIdx.x, tx = tile % P.ntx, ty = tile / P.ntx;
    const int x0 = tx * TRK_TW, y0 = ty * TRK_TH;
    TRK_T(0);
    s_val[tid] = P.val[tid];
    if (tid == 0) s_nslots = 0;
    __syncthreads();
    TRK_T(1);

    // ---- 1. point operations: TRK_NH units of four pixels per thread (rows ly, ly + 16) ---------------------------------------
    const int ux = (tid & 15) * 4;
    unsigned seedbits[TRK_NH] = {};                               // bit k: pixel k of the unit has mhi == ts
    int mine = 0;                                                  // does this thread hold any pixel with history?
#pragma unroll
    for (int half = 0; half < TRK_NH; half++) {
        const int ly = (tid >> 4) + half * 16, y = y0 + ly, x = x0 + ux, li = ly * TRK_TW + ux;
        int g[4] = {0, 0, 0, 0};
        unsigned hv[4] = {0, 0, 0, 0};
        int pv[4] = {0, 0, 0, 0};
        const bool row_ok = y < P.h;
        const bool full = row_ok && x + 3 < P.w;
        if (FMT == 0 && P.vec && full) {
            const uint4 px = *reinterpret_cast<const uint4 *>(P.src.p0 + (size_t)y * P.src.s0 + 4 * x);
            const unsigned w4[4] = {px.x, px.y, px.z, px.w};
#pragma unroll
            for (int k = 0; k < 4; k++) g[k] = trk_gray(w4[k] & 255, (w4[k] >> 8) & 255, (w4[k] >> 16) & 255);
            const unsigned p4 = *reinterpret_cast<const unsigned *>(P.prev + (size_t)y * P.w + x);
            const unsigned h4 = P.first ? 0u : *reinterpret_cast<const unsigned *>(P.hist + (size_t)y * P.w + x);
#pragma unroll
            for (int k = 0; k < 4; k++) { pv[k] = (p4 >> (8 * k)) & 255; hv[k] = (h4 >> (8 * k)) & 255; }
        } else if (row_ok) {
#pragma unroll
            for (int k = 0; k < 4; k++) {
                if (x + k >= P.w) break;
                if (FMT == 0) {
                    const uchar4 px = *reinterpret_cast<const uchar4 *>(P.src.p0 + (size_t)y * P.src.s0 + 4 * (x + k));
                    g[k] = trk_gray(px.x, px.y, px.z);
                } else {
                    int c3[3];
                    yuv_pixel(P.src, yuv_chroma<FMT == 0 ? 1 : FMT>(P.src, x + k, y), x + k, y, c3);
                    g[k] = trk_gray(c3[0], c3[1], c3[2]);
                }
                pv[k] = P.prev[(size_t)y * P.w + x + k];
                hv[k] = P.first ? 0u : P.hist[(size_t)y * P.w + x + k];
            }
        }
        unsigned nh[4];
        float m[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const bool in = row_ok && x + k < P.w;
            const bool silh = abs(g[k] - pv[k]) > P.thr;                                  // absdiff + threshold(.., BINARY)
            nh[k] = !in ? 0u : silh ? (unsigned)P.cur : (s_val[hv[k]] != 0.f ? hv[k] : 0u);   // updateMotionHistory
            m[k] = s_val[nh[k]];
            // history index P.cur <=> mhi == ts (equal float values share an index; value 0: no seeds at all)
            if (in && nh[k] == (unsigned)P.cur && m[k] != 0.f) seedbits[half] |= 1u << k;
        }
        if (row_ok) {
            if (P.vec && full) {
                *reinterpret_cast<unsigned *>(P.prev + (size_t)y * P.w + x) = (unsigned)g[0] | ((unsigned)g[1] << 8) | ((unsigned)g[2] << 16) | ((unsigned)g[3] << 24);
                if (!P.first) *reinterpret_cast<unsigned *>(P.hist + (size_t)y * P.w + x) = nh[0] | (nh[1] << 8) | (nh[2] << 16) | (nh[3] << 24);
            } else {
                for (int k = 0; k < 4 && x + k < P.w; k++) {
                    P.prev[(size_t)y * P.w + x + k] = (uint8_t)g[k];
                    if (!P.first) P.hist[(size_t)y * P.w + x + k] = (uint8_t)nh[k];
                }
            }
        }
        // ---- 2a. labels, pre-linked inside the unit ---------------------------------------------------------------------
        int lab = TRK_NONE;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            s_a.m[li + k] = m[k];
            mine |= m[k] != 0.f;
            lab = m[k] == 0.f ? TRK_NONE : (k > 0 && lab != TRK_NONE && trk_joined(m[k - 1], m[k])) ? lab : li + k;
            s_lab[li + k] = lab;
        }
    }
    if (P.first) return;                                           // the first frame only primes img_prev (:360)
    // a tile without any history (most of a frame, most of the time) has nothing to label: it only publishes an empty
    // perimeter and takes part in the edge and completion protocol
    const bool empty = !__syncthreads_or(mine);
    TRK_T(2);
    int root[TRK_NH][4];
#pragma unroll
    for (int half = 0; half < TRK_NH; half++)
#pragma unroll
        for (int k = 0; k < 4; k++) root[half][k] = TRK_NONE;
    if (!empty) {

    // ---- 2b. unions: along the rows first, then between rows, each followed by pointer jumping -----------------------------
    // Links point at smaller indices, so a blob that fills the tile would leave chains of up to 16 + 32 links (units of a
    // row, rows of the tile) and every find of the next phase would walk them through shared memory (measured: 31 000
    // cycles for the flatten of such a tile).  Pointer jumping (label <- label of label until nothing moves) turns the
    // forest into stars in log2(chain) block-wide steps; roots never move, so it may run between the two union phases.
    auto jump = [&]() {
        for (;;) {
            int moved = 0;
#pragma unroll
            for (int half = 0; half < TRK_NH; half++) {
                const int li = ((tid >> 4) + half * 16) * TRK_TW + ux;
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const int p = ((volatile int *)s_lab)[li + k];
                    if (p == TRK_NONE) continue;
                    const int pp = ((volatile int *)s_lab)[p];
                    if (pp != p) { s_lab[li + k] = pp; moved = 1; }
                }
            }
            if (!__syncthreads_or(moved)) break;
        }
    };
#pragma unroll
    for (int half = 0; half < TRK_NH; half++) {
        const int li = ((tid >> 4) + half * 16) * TRK_TW + ux;
        if (ux + 4 < TRK_TW && trk_joined(s_a.m[li + 3], s_a.m[li + 4])) trk_union(s_lab, li + 3, li + 4);
    }
    __syncthreads();
    jump();
#pragma unroll
    for (int half = 0; half < TRK_NH; half++) {
        const int ly = (tid >> 4) + half * 16, li = ly * TRK_TW + ux;
        if (ly + 1 < TRK_TH) {
            // was the vertical edge one pixel to the left joined?  (also across the unit boundary: inside a blob only the
            // first column of every row pair is linked, one union per pair of runs instead of one per pixel)
            bool prev_v = ux > 0 && trk_joined(s_a.m[li - 1], s_a.m[li - 1 + TRK_TW]);
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const float a = s_a.m[li + k], b = s_a.m[li + k + TRK_TW];
                const bool v = trk_joined(a, b);
                // skip an edge that closes a 2x2 cycle whose other three edges are joined
                const bool redundant = v && (k > 0 || ux > 0) && prev_v && trk_joined(s_a.m[li + k - 1], a) && trk_joined(s_a.m[li + k - 1 + TRK_TW], b);
                if (v && !redundant) trk_union(s_lab, li + k, li + k + TRK_TW);
                prev_v = v;
            }
        }
    }
    __syncthreads();
    TRK_T(3);
    // ---- 2c. flatten -----------------------------------------------------------------------------------------------------
    jump();
#pragma unroll
    for (int half = 0; half < TRK_NH; half++) {
        const int li = ((tid >> 4) + half * 16) * TRK_TW + ux;
#pragma unroll
        for (int k = 0; k < 4; k++) root[half][k] = s_lab[li + k];
    }
    __syncthreads();                                               // every find is done: s_a.m is dead, s_lab may be rewritten
#pragma unroll
    for (int half = 0; half < TRK_NH; half++) {
        const int ly = (tid >> 4) + half * 16, li = ly * TRK_TW + ux;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            s_lab[li + k] = root[half][k];
            s_a.minx[li + k] = TRK_TW; s_maxx[li + k] = -1; s_maxy[li + k] = -1; s_seed[li + k] = TRK_NONE;
        }
    }
    __syncthreads();
    TRK_T(4);

    // ---- 3. per-root reductions: runs of equal root inside a unit first, lanes with the same root next, then one atomic ---
#pragma unroll
    for (int half = 0; half < TRK_NH; half++) {
        const int ly = (tid >> 4) + half * 16, li = ly * TRK_TW + ux;
#pragma unroll
        for (int k = 0; k < 4; k++) {                              // round k: the run of equal roots that STARTS at pixel k, if any
            const int rk = root[half][k];
            const bool start = rk != TRK_NONE && (k == 0 || rk != root[half][k - 1]);
            int mnx = ux + k, mxx = ux + k, sd = ((seedbits[half] >> k) & 1u) ? li + k : TRK_NONE;
            bool cont = start;
#pragma unroll
            for (int j = k + 1; j < 4; j++) {
                cont = cont && root[half][j] == rk;
                if (cont) { mxx = ux + j; if (sd == TRK_NONE && ((seedbits[half] >> j) & 1u)) sd = li + j; }
            }
            if (!start) { mnx = TRK_TW; mxx = -1; sd = TRK_NONE; }
            const int mxy0 = start ? ly : -1;
            // a warp covers two 64-pixel rows: inside a blob every run of the round belongs to ONE component, and the whole
            // warp reduces with the full-mask REDUX (the per-group form of __reduce_*_sync is emulated and slow)
            const unsigned has = __ballot_sync(0xffffffffu, start);
            if (has) {
                const int leader = __ffs(has) - 1;
                const int r0 = __shfl_sync(0xffffffffu, rk, leader);
                if (__all_sync(0xffffffffu, !start || rk == r0)) {
                    const int a = __reduce_min_sync(0xffffffffu, mnx), b = __reduce_max_sync(0xffffffffu, mxx);
                    const int c = __reduce_max_sync(0xffffffffu, mxy0), d = __reduce_min_sync(0xffffffffu, sd);
                    if (lane == leader) {
                        atomicMin(&s_a.minx[r0], a); atomicMax(&s_maxx[r0], b); atomicMax(&s_maxy[r0], c);
                        if (d != TRK_NONE) atomicMin(&s_seed[r0], d);
                    }
                } else if (start) {
                    atomicMin(&s_a.minx[rk], mnx); atomicMax(&s_maxx[rk], mxx); atomicMax(&s_maxy[rk], mxy0);
                    if (sd != TRK_NONE) atomicMin(&s_seed[rk], sd);
                }
            }
        }
    }
    __syncthreads();
    TRK_T(5);

    // ---- 4. roots: final inside the tile, or a slot of the perimeter table ------------------------------------------------
    int *const parent = P.parent + (size_t)tile * TRK_SLOTS;
#pragma unroll
    for (int half = 0; half < TRK_NH; half++) {
        const int ly = (tid >> 4) + half * 16, li = ly * TRK_TW + ux;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int i = li + k;
            if (root[half][k] != i) continue;
            const int mnx = s_a.minx[i], mxx = s_maxx[i], mxy = s_maxy[i], sd = s_seed[i];
            const int gseed = sd == TRK_NONE ? TRK_NONE : (y0 + sd / TRK_TW) * P.w + x0 + (sd % TRK_TW);
            const bool edge = mnx == 0 || mxx == TRK_TW - 1 || ly == 0 || mxy == TRK_TH - 1;      // a root is its component's first row
            if (edge) {
                const int s = atomicAdd(&s_nslots, 1);
                P.bbox[(size_t)tile * TRK_SLOTS + s] = make_int4(x0 + mnx, y0 + ly, x0 + mxx, y0 + mxy);
                P.bseed[(size_t)tile * TRK_SLOTS + s] = gseed;
                parent[s] = tile * TRK_SLOTS + s;
                s_maxx[i] = s;                                     // slot of this root, read back below
            } else if (gseed != TRK_NONE) {
                const int pos = atomicAdd(&P.counters[0], 1);
                if (pos < TRK_MAX_COMPONENTS) { P.keys[pos] = gseed; P.rects[pos] = make_int4(x0 + mnx, y0 + ly, mxx - mnx + 1, mxy - ly + 1); }
            }
        }
    }
    __syncthreads();
    } else { TRK_T(3); TRK_T(4); TRK_T(5); }
    if (tid < TRK_PERIM) {
        const int r = s_lab[trk_perim_px(tid)];
        P.bslot[(size_t)tile * TRK_PERIM + tid] = r == TRK_NONE ? (unsigned short)0xffff : (unsigned short)s_maxx[r];
    }
    if (tid == 0) { P.bcount[tile] = s_nslots; s_base = s_nslots ? atomicAdd(&P.counters[2], s_nslots) : 0; }
    __syncthreads();
    for (int s2 = tid; s2 < s_nslots; s2 += blockDim.x) P.slotlist[s_base + s2] = tile * TRK_SLOTS + s2;     // for the last block
    __threadfence();
    __syncthreads();

    TRK_T(6);
    // ---- 5. stitch the edges this tile is the second to reach ---------------------------------------------------------------
    const int nh_edges = (P.ntx - 1) * P.nty;
    if (tid < 4) {
        int e = -1;
        if (tid == 0 && tx + 1 < P.ntx) e = ty * (P.ntx - 1) + tx;                        // right
        if (tid == 1 && tx > 0) e = ty * (P.ntx - 1) + tx - 1;                            // left
        if (tid == 2 && ty + 1 < P.nty) e = nh_edges + ty * P.ntx + tx;                   // below
        if (tid == 3 && ty > 0) e = nh_edges + (ty - 1) * P.ntx + tx;                     // above
        const bool second = e >= 0 && atomicAdd(&P.edge_flag[e], 1) == 1;
        if (second) P.edge_flag[e] = 0;                            // both tiles have been here: re-armed for the next frame
        s_edges[tid] = second ? 1 : 0;
    }
    __syncthreads();
    TRK_T(7);
    if (s_edges[0] || s_edges[1] || s_edges[2] || s_edges[3]) {
        __threadfence();                                           // the other tile published before it arrived at the edge
        if (s_edges[0]) trk_stitch(P, s_val, tile, tile + 1, 0);
        if (s_edges[1]) trk_stitch(P, s_val, tile - 1, tile, 0);
        if (s_edges[2]) trk_stitch(P, s_val, tile, tile + P.ntx, 1);
        if (s_edges[3]) trk_stitch(P, s_val, tile - P.ntx, tile, 1);
        __threadfence();
    }
    __syncthreads();
    TRK_T(8);
    if (tid == 0) s_last = atomicAdd(&P.counters[1], 1) == P.ntx * P.nty - 1;
    __syncthreads();
    TRK_T(9);
    if (!s_last) return;

    // ---- 6. the last block: fold slot records into their roots, collect, order ------------------------------------------------
    // one block from here on: __syncthreads() orders its own global accesses, the fence below is the acquire side of the
    // other blocks' releases
    __threadfence();
    const int nused = ((volatile int *)P.counters)[2];
    for (int i = tid; i < nused; i += blockDim.x) {
        const int gidx = __ldcg(P.slotlist + i), r = trk_find(P.parent, gidx);
        if (r == gidx) continue;
        const int4 b = __ldcg(P.bbox + gidx);
        int *rb = reinterpret_cast<int *>(P.bbox + r);
        atomicMin(rb + 0, b.x); atomicMin(rb + 1, b.y); atomicMax(rb + 2, b.z); atomicMax(rb + 3, b.w);
        const int sd = __ldcg(P.bseed + gidx);
        if (sd != TRK_NONE) atomicMin(P.bseed + r, sd);
    }
    __syncthreads();
    for (int i = tid; i < nused; i += blockDim.x) {
        const int gidx = __ldcg(P.slotlist + i);
        if (((volatile int *)P.parent)[gidx] != gidx) continue;
        const int sd = ((volatile int *)P.bseed)[gidx];
        if (sd == TRK_NONE) continue;
        const int pos = atomicAdd(&P.counters[0], 1);
        if (pos < TRK_MAX_COMPONENTS) {
            const volatile int *b = reinterpret_cast<volatile int *>(P.bbox + gidx);
            P.keys[pos] = sd;
            P.rects[pos] = make_int4(b[0], b[1], b[2] - b[0] + 1, b[3] - b[1] + 1);
        }
    }
    __syncthreads();
    const int total = ((volatile int *)P.counters)[0], n = min(total, TRK_MAX_COMPONENTS);
    // rank by first seed pixel (keys are distinct); up to a tile's worth of keys is ranked out of shared memory
    const bool in_smem = n <= TRK_NPX;
    if (in_smem) {
        for (int i = tid; i < n; i += blockDim.x) s_lab[i] = __ldcg(P.keys + i);
        __syncthreads();
    }
    for (int i = tid; i < n; i += blockDim.x) {
        const int key = in_smem ? s_lab[i] : __ldcg(P.keys + i);
        int rank = 0;
        if (in_smem) for (int j = 0; j < n; j++) rank += s_lab[j] < key;
        else for (int j = 0; j < n; j++) rank += __ldcg(P.keys + j) < key;
        const int4 r = __ldcg(P.rects + i);
        P.out[1 + rank] = r;
        if (P.hout && rank < 1024) P.hout[1 + rank] = r;
    }
    if (tid == 0) {
        P.out[0] = make_int4(total, 0, 0, 0);
        if (P.hout) P.hout[0] = make_int4(total, 0, 0, 0);
        P.counters[0] = 0; P.counters[1] = 0; P.counters[2] = 0;
    }
    TRK_T(10);
}

size_t tracker_scratch_bytes(int w, int h, TrkLayout *lo)
{
    const int ntx = (w + TRK_TW - 1) / TRK_TW, nty = (h + TRK_TH - 1) / TRK_TH, nt = ntx * nty;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o += (bytes + 255) & ~(size_t)255; return at; };
    lo->ntx = ntx; lo->nty = nty;
    lo->bbox = take((size_t)nt * TRK_SLOTS * sizeof(int4));
    lo->rects = take((size_t)TRK_MAX_COMPONENTS * sizeof(int4));
    lo->out = take((size_t)(1 + TRK_MAX_COMPONENTS) * sizeof(int4));
    lo->bseed = take((size_t)nt * TRK_SLOTS * sizeof(int));
    lo->parent = take((size_t)nt * TRK_SLOTS * sizeof(int));
    lo->slotlist = take((size_t)nt * TRK_SLOTS * sizeof(int));
    lo->bcount = take((size_t)nt * sizeof(int));
    lo->keys = take((size_t)TRK_MAX_COMPONENTS * sizeof(int));
    lo->bslot = take((size_t)nt * TRK_PERIM * sizeof(unsigned short));
    lo->zero_begin = o;                                             // counters and edge flags start (and are left) at zero
    lo->counters = take(4 * sizeof(int));
    lo->edge_flag = take((size_t)(2 * nt + 1) * sizeof(int));
    lo->zero_end = o;
    return o;
}

cudaError_t launch_tracker(nv_ctx *ctx, int fmt, const SrcPlanes &src, int w, int h, int first, int thr, int cur, const float *val256,
                           int *nlaunch)
{
    const TrkLayout &lo = ctx->trk_lo;
    uint8_t *base = ctx->d_trk_scratch;
    TrkParams P;
    P.src = src; P.w = w; P.h = h; P.first = first; P.thr = thr; P.cur = cur; P.ntx = lo.ntx; P.nty = lo.nty;
    P.vec = fmt == NV_FMT_BGR && (w % 4) == 0 && (src.s0 % 16) == 0 && ((uintptr_t)src.p0 % 16) == 0;
    P.prev = ctx->d_trk_prev; P.hist = ctx->d_trk_hist;
    P.bslot = reinterpret_cast<unsigned short *>(base + lo.bslot); P.bcount = reinterpret_cast<int *>(base + lo.bcount);
    P.bbox = reinterpret_cast<int4 *>(base + lo.bbox); P.bseed = reinterpret_cast<int *>(base + lo.bseed);
    P.slotlist = reinterpret_cast<int *>(base + lo.slotlist);
    P.parent = reinterpret_cast<int *>(base + lo.parent); P.edge_flag = reinterpret_cast<int *>(base + lo.edge_flag);
    P.counters = reinterpret_cast<int *>(base + lo.counters); P.keys = reinterpret_cast<int *>(base + lo.keys);
    P.rects = reinterpret_cast<int4 *>(base + lo.rects); P.out = reinterpret_cast<int4 *>(base + lo.out);
    P.hout = reinterpret_cast<int4 *>(ctx->h_trk);
    for (int i = 0; i < 256; i++) P.val[i] = val256[i];
    const int nt = lo.ntx * lo.nty;
    cudaStream_t st = ctx->stream;
    if (fmt == NV_FMT_BGR) k_trk_fused<0><<<nt, 256, 0, st>>>(P);               // interleaved: BGRA here
    else if (fmt == NV_FMT_I420) k_trk_fused<1><<<nt, 256, 0, st>>>(P);
    else if (fmt == NV_FMT_NV12) k_trk_fused<2><<<nt, 256, 0, st>>>(P);
    else if (fmt == NV_FMT_NV21) k_trk_fused<3><<<nt, 256, 0, st>>>(P);
    else return cudaErrorInvalidValue;
    (*nlaunch)++;
    return cudaGetLastError();
}
