// cascade_eval.cuh — one weak classifier / one stage at one window, in the reference's arithmetic (SURVEY.md A.6).
// Shared by the cascade kernels (kernels_cascade.cu) and the score pass of the candidate sort (kernels_group.cu).
#pragma once
#include "internal.h"

struct LevelView {
    const uint32_t *sum;
    int pitch, plane, ys;
};

__device__ __forceinline__ int corner(const LevelView &v, int dx, int dy)
{
    return dy * v.pitch + (v.ys == 2 ? (dx & 1) * v.plane + (dx >> 1) : dx);
}

__device__ __forceinline__ int rect_sum(const uint32_t *__restrict__ wb, const LevelView &v, uint32_t packed)
{
    int x = packed & 255, y = (packed >> 8) & 255, w = (packed >> 16) & 255, h = packed >> 24;
    uint32_t a = __ldg(wb + corner(v, x, y)), b = __ldg(wb + corner(v, x + w, y));
    uint32_t c = __ldg(wb + corner(v, x, y + h)), d = __ldg(wb + corner(v, x + w, y + h));
    return (int)(a - b - c + d);
}

struct StumpRegs {
    uint32_t r0, r1, r2;
    float w0, w1, w2, thr, left, right;
};

__device__ __forceinline__ StumpRegs load_stump(const DevStump *__restrict__ s)
{
    const uint4 *p = reinterpret_cast<const uint4 *>(s);
    uint4 a = __ldg(p), b = __ldg(p + 1), c = __ldg(p + 2);
    StumpRegs o;
    o.r0 = a.x; o.r1 = a.y; o.r2 = a.z;
    o.w0 = __uint_as_float(a.w); o.w1 = __uint_as_float(b.x); o.w2 = __uint_as_float(b.y);
    o.thr = __uint_as_float(b.z); o.left = __uint_as_float(b.w); o.right = __uint_as_float(c.x);
    return o;
}

// value of one weak classifier at the window whose top-left integral element is wb
__device__ __forceinline__ float stump_leaf(const uint32_t *__restrict__ wb, const LevelView &v, const StumpRegs &s,
                                            float vnf)
{
    float f = __fmul_rn(s.w0, __int2float_rn(rect_sum(wb, v, s.r0)));
    f = __fadd_rn(f, __fmul_rn(s.w1, __int2float_rn(rect_sum(wb, v, s.r1))));
    if (s.w2 != 0.f) f = __fadd_rn(f, __fmul_rn(s.w2, __int2float_rn(rect_sum(wb, v, s.r2))));
    f = __fmul_rn(f, vnf);
    return f < s.thr ? s.left : s.right;
}

__device__ __forceinline__ float gen_feature(const GenModel &g, int f, const uint32_t *__restrict__ wb, const LevelView &v,
                                             const uint32_t *__restrict__ tb, int tp)
{
    const GenFeat ft = g.feat[f];
    float val = 0.f;
#pragma unroll
    for (int k = 0; k < 3; k++) {
        if (k == 2 && ft.w[2] == 0.f) break;
        uint32_t pr = ft.r[k];
        int rs;
        if (ft.tilted) {                                         // (x, y), (x - h, y + h), (x + w, y + w), (x + w - h, y + w + h)
            int x = pr & 255, y = (pr >> 8) & 255, w = (pr >> 16) & 255, h = pr >> 24;
            rs = (int)(__ldg(tb + y * tp + x) - __ldg(tb + (y + h) * tp + x - h) - __ldg(tb + (y + w) * tp + x + w) +
                       __ldg(tb + (y + w + h) * tp + x + w - h));
        } else
            rs = rect_sum(wb, v, pr);
        float t = __fmul_rn(ft.w[k], __int2float_rn(rs));
        val = k == 0 ? t : __fadd_rn(val, t);
    }
    return val;
}

// LBP feature (OpenCV LBPEvaluator::OptFeature::calc): the cell rect spans a 3 x 3 grid of cells; the eight outer cell
// sums are compared (>=) with the centre one, clockwise from the top-left, most significant bit first.
__device__ __forceinline__ int lbp_code(const GenModel &g, int f, const uint32_t *__restrict__ wb, const LevelView &v)
{
    const uint32_t pr = g.feat[f].r[0];
    const int x = pr & 255, y = (pr >> 8) & 255, w = (pr >> 16) & 255, h = pr >> 24;
    uint32_t p[4][4];
#pragma unroll
    for (int j = 0; j < 4; j++)
#pragma unroll
        for (int i = 0; i < 4; i++) p[j][i] = __ldg(wb + corner(v, x + i * w, y + j * h));
    auto cell = [&](int j, int i) { return (int)(p[j][i] - p[j][i + 1] - p[j + 1][i] + p[j + 1][i + 1]); };
    const int c = cell(1, 1);
    return (cell(0, 0) >= c ? 128 : 0) | (cell(0, 1) >= c ? 64 : 0) | (cell(0, 2) >= c ? 32 : 0) | (cell(1, 2) >= c ? 16 : 0) |
           (cell(2, 2) >= c ? 8 : 0) | (cell(2, 1) >= c ? 4 : 0) | (cell(2, 0) >= c ? 2 : 0) | (cell(1, 0) >= c ? 1 : 0);
}

// Stage sum of trees [t0, t1) in XML order, leaves accumulated in double.  Haar models: OpenCV's predictOrdered (float
// feature value times the variance factor against the node threshold); LBP models (g.subset != nullptr): OpenCV's
// predictCategorical — the node's feature code goes left when its bit is set in the node's 256-bit subset.
__device__ __forceinline__ double gen_stage_sum(const GenModel &g, int t0, int t1, const uint32_t *__restrict__ wb,
                                                const LevelView &v, const uint32_t *__restrict__ tb, int tp, float vnf)
{
    double tmp = 0.;
    for (int t = t0; t < t1; t++) {
        int2 tr = g.tree[t];                                     // first node, first leaf
        int idx = 0;
        do {
            int4 n = g.node[tr.x + idx];                         // feature, threshold bits, left, right
            if (g.subset) {
                const int code = lbp_code(g, n.x, wb, v);
                idx = (__ldg(g.subset + (size_t)(tr.x + idx) * 8 + (code >> 5)) >> (code & 31)) & 1u ? n.z : n.w;
                continue;
            }
            float val = __fmul_rn(gen_feature(g, n.x, wb, v, tb, tp), vnf);
            idx = val < __int_as_float(n.y) ? n.z : n.w;
        } while (idx > 0);
        tmp = __dadd_rn(tmp, (double)g.leaf[tr.y - idx]);
    }
    return tmp;
}
