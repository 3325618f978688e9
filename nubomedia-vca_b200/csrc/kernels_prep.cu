// kernels_prep.cu — K1/K2/K3: colour conversion, cv::resize(INTER_LINEAR), equalizeHist pieces, flip.
// Arithmetic follows OpenCV 4.13 bit-exactly (SURVEY.md A.1–A.3; oracle/nubo_oracle.c is the checker).
// Reference call sites: kmsfacedetect.cpp:805-807, kmseyedetect.cpp:949-964, kmsmouthdetect.cpp:836-853,
// kmsnosedetect.cpp:834-851, kmseardetect.cpp:786-800, gstnubotracker.cpp:356.
#include <math.h>

#include "internal.h"

// ------------------------------------------------------------------------------------------------
// host: coefficient tables of cv::resize(INTER_LINEAR) for u8 (11-bit fixed point)
// ------------------------------------------------------------------------------------------------
static inline int sat_short(int v) { return v < -32768 ? -32768 : (v > 32767 ? 32767 : v); }

void build_resize_tables(int sw, int sh, int dw, int dh, std::vector<int> &tab)
{
    tab.clear();
    if (sw == dw && sh == dh) { tab.push_back(RT_COPY); return; }
    if (sw == 2 * dw && sh == 2 * dh) { tab.push_back(RT_BOX2); return; }   // INTER_AREA fast path
    tab.resize(1 + 2 * (size_t)dw + 3 * (size_t)dh);
    tab[0] = RT_LINEAR;
    int *xofs = &tab[1], *xa = xofs + dw, *y0 = xa + dw, *y1 = y0 + dh, *yb = y1 + dh;
    double scale_x = 1.0 / ((double)dw / sw), scale_y = 1.0 / ((double)dh / sh);
    for (int dx = 0; dx < dw; dx++) {
        float fx = (float)((dx + 0.5) * scale_x - 0.5);
        int sx = (int)floorf(fx);
        fx -= sx;
        if (sx < 0) { fx = 0; sx = 0; }
        if (sx >= sw - 1) { fx = 0; sx = sw - 1; }
        int a0 = sat_short((int)lrintf((1.f - fx) * 2048)), a1 = sat_short((int)lrintf(fx * 2048));
        xofs[dx] = sx;
        xa[dx] = (a0 & 0xFFFF) | (a1 << 16);
    }
    for (int dy = 0; dy < dh; dy++) {
        float fy = (float)((dy + 0.5) * scale_y - 0.5);
        int sy = (int)floorf(fy);
        fy -= sy;
        // vertical coefficients keep their fraction; only the row indices are clamped
        int b0 = sat_short((int)lrintf((1.f - fy) * 2048)), b1 = sat_short((int)lrintf(fy * 2048));
        y0[dy] = sy < 0 ? 0 : (sy > sh - 1 ? sh - 1 : sy);
        y1[dy] = sy + 1 < 0 ? 0 : (sy + 1 > sh - 1 ? sh - 1 : sy + 1);
        yb[dy] = (b0 & 0xFFFF) | (b1 << 16);
    }
}

// ------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int gray_of(int b, int g, int r)
{
    return (b * 3735 + g * 19235 + r * 9798 + 16384) >> 15;     // A.1, 15-bit coefficients
}

__device__ __forceinline__ int lin_tap(const uint8_t *__restrict__ r0, const uint8_t *__restrict__ r1, int i0, int i1,
                                       int a0, int a1, int b0, int b1)
{
    int h0 = r0[i0] * a0 + r0[i1] * a1;
    int h1 = r1[i0] * a0 + r1[i1] * a1;
    return (((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2;       // A.2 vertical pass
}

// histogram -> equalizeHist LUT (A.3), by one block of 256 threads: lut[k] = sat_u8(rint((float)(cum[k] - cum[i0]) *
// (255.f / (total - hist[i0])))).  cum / s_i0: shared scratch of the caller.
__device__ __forceinline__ uint8_t lut_entry(int t, int hv, int total, int *cum, int *s_i0)
{
    if (t == 0) *s_i0 = 256;
    cum[t] = hv;
    __syncthreads();
    if (hv) atomicMin(s_i0, t);
    for (int d = 1; d < 256; d <<= 1) {         // Hillis-Steele inclusive scan
        int v = t >= d ? cum[t - d] : 0;
        __syncthreads();
        cum[t] += v;
        __syncthreads();
    }
    const int i0 = *s_i0;
    if (i0 >= 256) return (uint8_t)t;                                  // empty image: identity
    const int h0 = cum[i0] - (i0 ? cum[i0 - 1] : 0);
    if (h0 == total) return (uint8_t)i0;                               // constant image
    if (t <= i0) return 0;
    const float scale = __fdiv_rn(255.f, __int2float_rn(total - h0));
    const int v = __float2int_rn(__fmul_rn(__int2float_rn(cum[t] - cum[i0]), scale));
    return (uint8_t)min(max(v, 0), 255);
}

// End of a face-prep kernel: flush the block's histogram; with `lut` set, the block that finishes LAST (a ticket in
// hist[256]) turns the complete histogram into the LUT and clears histogram and ticket for the next frame — what a k_lut
// does as a launch of its own (one block, ~4 us of a small call's chain) when the histogram comes from elsewhere.
// BATCH: one image per gridDim.y row; the ticket counts that image's blocks only.
template <bool BATCH = false>
__device__ __forceinline__ void prep_finish(int tid, int *sh_hist, int *__restrict__ hist, uint8_t *__restrict__ lut, int total)
{
    __shared__ int s_i0, s_last;
    __syncthreads();
    if (sh_hist[tid]) atomicAdd(&hist[tid], sh_hist[tid]);
    if (!lut) return;
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(&hist[256], 1) == (int)(BATCH ? gridDim.x : gridDim.x * gridDim.y) - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    const int hv = __ldcg(&hist[tid]);
    lut[tid] = lut_entry(tid, hv, total, sh_hist, &s_i0);
    hist[tid] = 0;
    if (tid == 0) hist[256] = 0;
}

// K1+K2 fused for the face element: resize the BGR(A) frame (3 channels computed), convert to gray,
// accumulate the histogram equalizeHist needs.  One thread per output pixel.
// Blocks walk the 32x8-pixel output tiles with a grid stride (the launchers size the grid to a few blocks per SM): the
// shared histogram is flushed once per block, so the global histogram sees a few hundred atomics per bin and frame
// instead of one per bin and tile (8100 tiles on a 1080p frame).
// BATCH: image blockIdx.y reads its frame from srcs[blockIdx.y] and owns gray, histogram (+ ticket) and LUT at
// blockIdx.y times the strides.
template <bool BATCH>
__global__ void __launch_bounds__(256)
k_face_prep(const uint8_t *__restrict__ src, int sw, int sh, int sstride, int cn, uint8_t *__restrict__ gray, int dw,
            int dh, const int *__restrict__ rtab, int *__restrict__ hist, uint8_t *__restrict__ lut,
            const uint8_t *const *__restrict__ srcs = nullptr, size_t gray_stride = 0)
{
    __shared__ int sh_hist[256];
    if (BATCH) {
        src = srcs[blockIdx.y];
        gray += blockIdx.y * gray_stride; hist += blockIdx.y * NV_HIST_STRIDE; lut += blockIdx.y * 256;
    }
    int tid = threadIdx.y * 32 + threadIdx.x;
    sh_hist[tid] = 0;
    __syncthreads();
    const int tx_n = (dw + 31) / 32, ntiles = tx_n * ((dh + 7) / 8), mode = rtab[0];
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        int x = (t % tx_n) * 32 + threadIdx.x, y = (t / tx_n) * 8 + threadIdx.y;
        if (x >= dw || y >= dh) continue;
        int g;
        if (mode == RT_COPY) {
            const uint8_t *p = src + (size_t)y * sstride + x * cn;
            g = gray_of(p[0], p[1], p[2]);
        } else if (mode == RT_BOX2) {
            const uint8_t *p0 = src + (size_t)(2 * y) * sstride + 2 * x * cn, *p1 = p0 + sstride;
            int c3[3];
#pragma unroll
            for (int c = 0; c < 3; c++) c3[c] = (p0[c] + p0[c + cn] + p1[c] + p1[c + cn] + 2) >> 2;
            g = gray_of(c3[0], c3[1], c3[2]);
        } else {
            const int *xofs = rtab + 1, *xa = xofs + dw, *y0t = xa + dw, *y1t = y0t + dh, *ybt = y1t + dh;
            int sx = xofs[x], sx1 = min(sx + 1, sw - 1), xav = xa[x], ybv = ybt[y];
            int a0 = (short)(xav & 0xFFFF), a1 = xav >> 16, b0 = (short)(ybv & 0xFFFF), b1 = ybv >> 16;
            const uint8_t *r0 = src + (size_t)y0t[y] * sstride, *r1 = src + (size_t)y1t[y] * sstride;
            int c3[3];
#pragma unroll
            for (int c = 0; c < 3; c++) c3[c] = lin_tap(r0, r1, sx * cn + c, sx1 * cn + c, a0, a1, b0, b1);
            g = gray_of(c3[0], c3[1], c3[2]);
        }
        gray[(size_t)y * dw + x] = (uint8_t)g;
        atomicAdd(&sh_hist[g], 1);
    }
    prep_finish<BATCH>(tid, sh_hist, hist, lut, dw * dh);
}

// Vectorised forms of the two streaming modes (same size, exact 2x): a lane owns FOUR consecutive output pixels, reads
// its source bytes as aligned 32-bit words (12 bytes of BGR per row and output quad in copy mode, 24 in box mode) and
// writes one 32-bit word of gray; a warp's loads are one contiguous 384- / 768-byte run per source row.  Used when
// the output width is a multiple of 4 and pointer and stride are 4-byte aligned (GStreamer rows are), else the
// byte-per-lane kernel above runs.
__device__ __forceinline__ int byte_of(uint32_t w, int i) { return (int)((w >> (8 * i)) & 255u); }

template <int MODE, bool BATCH>
__global__ void __launch_bounds__(256)
k_face_prep_bgr4(const uint8_t *__restrict__ src, int sstride, uint8_t *__restrict__ gray, int dw, int dh,
                 int *__restrict__ hist, uint8_t *__restrict__ lut, const uint8_t *const *__restrict__ srcs = nullptr,
                 size_t gray_stride = 0)
{
    __shared__ int sh_hist[256];
    if (BATCH) {
        src = srcs[blockIdx.y];
        gray += blockIdx.y * gray_stride; hist += blockIdx.y * NV_HIST_STRIDE; lut += blockIdx.y * 256;
    }
    int tid = threadIdx.y * 32 + threadIdx.x;
    sh_hist[tid] = 0;
    __syncthreads();
    const int qw = dw >> 2, tx_n = (qw + 31) / 32, ntiles = tx_n * ((dh + 7) / 8);
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        int xq = (t % tx_n) * 32 + threadIdx.x, y = (t / tx_n) * 8 + threadIdx.y;
        if (xq >= qw || y >= dh) continue;
        int g[4];
        if (MODE == RT_COPY) {
            const uint32_t *p = reinterpret_cast<const uint32_t *>(src + (size_t)y * sstride) + 3 * xq;
            uint32_t w0 = __ldg(p), w1 = __ldg(p + 1), w2 = __ldg(p + 2);
            g[0] = gray_of(byte_of(w0, 0), byte_of(w0, 1), byte_of(w0, 2));
            g[1] = gray_of(byte_of(w0, 3), byte_of(w1, 0), byte_of(w1, 1));
            g[2] = gray_of(byte_of(w1, 2), byte_of(w1, 3), byte_of(w2, 0));
            g[3] = gray_of(byte_of(w2, 1), byte_of(w2, 2), byte_of(w2, 3));
        } else {
            const uint32_t *p0 = reinterpret_cast<const uint32_t *>(src + (size_t)(2 * y) * sstride) + 6 * xq;
            const uint32_t *p1 = reinterpret_cast<const uint32_t *>(src + (size_t)(2 * y + 1) * sstride) + 6 * xq;
            uint32_t a[6], b[6];
#pragma unroll
            for (int i = 0; i < 6; i++) { a[i] = __ldg(p0 + i); b[i] = __ldg(p1 + i); }
#pragma unroll
            for (int k = 0; k < 4; k++) {                     // output pixel k: source bytes 6k .. 6k+5 of both rows
                int c3[3];
#pragma unroll
                for (int c = 0; c < 3; c++) {
                    const int i0 = 6 * k + c, i1 = i0 + 3;
                    c3[c] = (byte_of(a[i0 >> 2], i0 & 3) + byte_of(a[i1 >> 2], i1 & 3) + byte_of(b[i0 >> 2], i0 & 3) +
                             byte_of(b[i1 >> 2], i1 & 3) + 2) >> 2;
                }
                g[k] = gray_of(c3[0], c3[1], c3[2]);
            }
        }
        *reinterpret_cast<uint32_t *>(gray + (size_t)y * dw + 4 * xq) =
            (uint32_t)g[0] | ((uint32_t)g[1] << 8) | ((uint32_t)g[2] << 16) | ((uint32_t)g[3] << 24);
#pragma unroll
        for (int k = 0; k < 4; k++) atomicAdd(&sh_hist[g[k]], 1);
    }
    prep_finish<BATCH>(tid, sh_hist, hist, lut, dw * dh);
}

// ---- 4:2:0 ingest (SURVEY §8f rank 4): the same block fed by I420 / NV12 / NV21 planes.  Every source pixel the
// resize touches is converted with cvtColor(COLOR_YUV2BGR_*)'s arithmetic (BT.601, 20-bit fixed point, saturated to
// u8 per pixel; oracle: ora_yuv420_to_bgr), so the result equals the reference block on the converted BGR frame.
// BATCH: image blockIdx.y takes its three plane pointers from planes[3 * blockIdx.y ..] (the strides in s are shared by
// all images) and owns gray, histogram (+ ticket) and LUT at blockIdx.y times the strides, as in k_face_prep.
template <int FMT, bool BATCH>
__global__ void __launch_bounds__(256)
k_face_prep_yuv(SrcPlanes s, int sw, int sh, uint8_t *__restrict__ gray, int dw, int dh, const int *__restrict__ rtab,
                int *__restrict__ hist, uint8_t *__restrict__ lut, const uint8_t *const *__restrict__ planes = nullptr,
                size_t gray_stride = 0)
{
    __shared__ int sh_hist[256];
    if (BATCH) {
        s.p0 = planes[3 * blockIdx.y]; s.p1 = planes[3 * blockIdx.y + 1]; s.p2 = planes[3 * blockIdx.y + 2];
        gray += blockIdx.y * gray_stride; hist += blockIdx.y * NV_HIST_STRIDE; lut += blockIdx.y * 256;
    }
    int tid = threadIdx.y * 32 + threadIdx.x;
    sh_hist[tid] = 0;
    __syncthreads();
    const int tx_n = (dw + 31) / 32, ntiles = tx_n * ((dh + 7) / 8), mode = rtab[0];
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        int x = (t % tx_n) * 32 + threadIdx.x, y = (t / tx_n) * 8 + threadIdx.y;
        if (x >= dw || y >= dh) continue;
        int g, c3[3];
        if (mode == RT_COPY) {
            yuv_pixel(s, yuv_chroma<FMT>(s, x, y), x, y, c3);
        } else if (mode == RT_BOX2) {                       // the four source pixels share one chroma sample
            YuvTerms t4 = yuv_chroma<FMT>(s, 2 * x, 2 * y);
            int a[3], b[3], c[3], d[3];
            yuv_pixel(s, t4, 2 * x, 2 * y, a);     yuv_pixel(s, t4, 2 * x + 1, 2 * y, b);
            yuv_pixel(s, t4, 2 * x, 2 * y + 1, c); yuv_pixel(s, t4, 2 * x + 1, 2 * y + 1, d);
#pragma unroll
            for (int k = 0; k < 3; k++) c3[k] = (a[k] + b[k] + c[k] + d[k] + 2) >> 2;
        } else {
            const int *xofs = rtab + 1, *xa = xofs + dw, *y0t = xa + dw, *y1t = y0t + dh, *ybt = y1t + dh;
            int sx = xofs[x], sx1 = min(sx + 1, sw - 1), xav = xa[x], ybv = ybt[y], sy0 = y0t[y], sy1 = y1t[y];
            int a0 = (short)(xav & 0xFFFF), a1 = xav >> 16, b0 = (short)(ybv & 0xFFFF), b1 = ybv >> 16;
            int p00[3], p01[3], p10[3], p11[3];
            yuv_pixel(s, yuv_chroma<FMT>(s, sx, sy0), sx, sy0, p00);   yuv_pixel(s, yuv_chroma<FMT>(s, sx1, sy0), sx1, sy0, p01);
            yuv_pixel(s, yuv_chroma<FMT>(s, sx, sy1), sx, sy1, p10);   yuv_pixel(s, yuv_chroma<FMT>(s, sx1, sy1), sx1, sy1, p11);
#pragma unroll
            for (int k = 0; k < 3; k++) {
                int h0 = p00[k] * a0 + p01[k] * a1, h1 = p10[k] * a0 + p11[k] * a1;
                c3[k] = (((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2;       // A.2 vertical pass
            }
        }
        g = gray_of(c3[0], c3[1], c3[2]);
        gray[(size_t)y * dw + x] = (uint8_t)g;
        atomicAdd(&sh_hist[g], 1);
    }
    prep_finish<BATCH>(tid, sh_hist, hist, lut, dw * dh);
}

// Vectorised 4:2:0 forms: a lane owns four consecutive output pixels.  Copy mode: 4 luma bytes (one word) and their
// two chroma samples; box mode: 2 x 8 luma bytes and four chroma samples.  Same alignment rule as k_face_prep_bgr4.
__device__ __forceinline__ YuvTerms yuv_terms(int u, int v)
{
    u -= 128; v -= 128;
    YuvTerms t;
    t.b = (1 << 19) + 2116026 * u;
    t.g = (1 << 19) - 852492 * v - 409993 * u;
    t.r = (1 << 19) + 1673527 * v;
    return t;
}
__device__ __forceinline__ void yuv_px(int yv, const YuvTerms &t, int c3[3])
{
    int yy = max(0, yv - 16) * 1220542;
    c3[0] = sat_u8((yy + t.b) >> 20); c3[1] = sat_u8((yy + t.g) >> 20); c3[2] = sat_u8((yy + t.r) >> 20);
}

template <int FMT, int MODE, bool BATCH>
__global__ void __launch_bounds__(256)
k_face_prep_yuv4(SrcPlanes s, uint8_t *__restrict__ gray, int dw, int dh, int *__restrict__ hist, uint8_t *__restrict__ lut,
                 const uint8_t *const *__restrict__ planes = nullptr, size_t gray_stride = 0)
{
    __shared__ int sh_hist[256];
    if (BATCH) {
        s.p0 = planes[3 * blockIdx.y]; s.p1 = planes[3 * blockIdx.y + 1]; s.p2 = planes[3 * blockIdx.y + 2];
        gray += blockIdx.y * gray_stride; hist += blockIdx.y * NV_HIST_STRIDE; lut += blockIdx.y * 256;
    }
    int tid = threadIdx.y * 32 + threadIdx.x;
    sh_hist[tid] = 0;
    __syncthreads();
    const int qw = dw >> 2, tx_n = (qw + 31) / 32, ntiles = tx_n * ((dh + 7) / 8);
    constexpr int NC = MODE == RT_COPY ? 2 : 4;              // chroma samples under a lane's source pixels
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        int xq = (t % tx_n) * 32 + threadIdx.x, y = (t / tx_n) * 8 + threadIdx.y;
        if (xq >= qw || y >= dh) continue;
        const int sx = MODE == RT_COPY ? 4 * xq : 8 * xq, sy = MODE == RT_COPY ? y : 2 * y;     // first source pixel
        int u[NC], v[NC];
        if (FMT == 1) {
            const uint8_t *pu = s.p1 + (size_t)(sy >> 1) * s.s1 + (sx >> 1), *pv = s.p2 + (size_t)(sy >> 1) * s.s2 + (sx >> 1);
            if (MODE == RT_COPY) {
                uint32_t wu = *reinterpret_cast<const uint16_t *>(pu), wv = *reinterpret_cast<const uint16_t *>(pv);
#pragma unroll
                for (int i = 0; i < NC; i++) { u[i] = byte_of(wu, i); v[i] = byte_of(wv, i); }
            } else {
                uint32_t wu = __ldg(reinterpret_cast<const uint32_t *>(pu)), wv = __ldg(reinterpret_cast<const uint32_t *>(pv));
#pragma unroll
                for (int i = 0; i < NC; i++) { u[i] = byte_of(wu, i); v[i] = byte_of(wv, i); }
            }
        } else {
            const uint32_t *pc = reinterpret_cast<const uint32_t *>(s.p1 + (size_t)(sy >> 1) * s.s1 + sx);
#pragma unroll
            for (int i = 0; i < NC / 2; i++) {
                uint32_t w = __ldg(pc + i);                  // two interleaved chroma pairs
                u[2 * i] = byte_of(w, FMT == 2 ? 0 : 1); v[2 * i] = byte_of(w, FMT == 2 ? 1 : 0);
                u[2 * i + 1] = byte_of(w, FMT == 2 ? 2 : 3); v[2 * i + 1] = byte_of(w, FMT == 2 ? 3 : 2);
            }
        }
        int g[4];
        if (MODE == RT_COPY) {
            uint32_t wy = __ldg(reinterpret_cast<const uint32_t *>(s.p0 + (size_t)sy * s.s0 + sx));
#pragma unroll
            for (int k = 0; k < 4; k++) {
                int c3[3];
                yuv_px(byte_of(wy, k), yuv_terms(u[k >> 1], v[k >> 1]), c3);
                g[k] = gray_of(c3[0], c3[1], c3[2]);
            }
        } else {
            const uint32_t *r0 = reinterpret_cast<const uint32_t *>(s.p0 + (size_t)sy * s.s0 + sx);
            const uint32_t *r1 = reinterpret_cast<const uint32_t *>(s.p0 + (size_t)(sy + 1) * s.s0 + sx);
            uint32_t a[2] = {__ldg(r0), __ldg(r0 + 1)}, b[2] = {__ldg(r1), __ldg(r1 + 1)};
#pragma unroll
            for (int k = 0; k < 4; k++) {                     // output pixel k: luma bytes 2k, 2k+1 of both rows, chroma k
                const YuvTerms tk = yuv_terms(u[k], v[k]);
                int p[4][3];
                yuv_px(byte_of(a[k >> 1], (2 * k) & 3), tk, p[0]); yuv_px(byte_of(a[k >> 1], (2 * k + 1) & 3), tk, p[1]);
                yuv_px(byte_of(b[k >> 1], (2 * k) & 3), tk, p[2]); yuv_px(byte_of(b[k >> 1], (2 * k + 1) & 3), tk, p[3]);
                int c3[3];
#pragma unroll
                for (int c = 0; c < 3; c++) c3[c] = (p[0][c] + p[1][c] + p[2][c] + p[3][c] + 2) >> 2;
                g[k] = gray_of(c3[0], c3[1], c3[2]);
            }
        }
        *reinterpret_cast<uint32_t *>(gray + (size_t)y * dw + 4 * xq) =
            (uint32_t)g[0] | ((uint32_t)g[1] << 8) | ((uint32_t)g[2] << 16) | ((uint32_t)g[3] << 24);
#pragma unroll
        for (int k = 0; k < 4; k++) atomicAdd(&sh_hist[g[k]], 1);
    }
    prep_finish<BATCH>(tid, sh_hist, hist, lut, dw * dh);
}

// BGR2GRAY(cvtColor(COLOR_YUV2BGR_*)) at full resolution: the first step of the nested elements on 4:2:0 frames
// (kmseyedetect.cpp:949 etc. after the conversion); one thread per pixel
template <int FMT>
__global__ void __launch_bounds__(256)
k_yuv2gray(SrcPlanes s, int w, int h, uint8_t *__restrict__ dst, int dstride)
{
    int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
    if (x >= w || y >= h) return;
    int c3[3];
    yuv_pixel(s, yuv_chroma<FMT>(s, x, y), x, y, c3);
    dst[(size_t)y * dstride + x] = (uint8_t)gray_of(c3[0], c3[1], c3[2]);
}

// cvtColor(COLOR_YUV2BGR_*) alone (parity tap of the ingest path); one thread per pixel
template <int FMT>
__global__ void __launch_bounds__(256)
k_yuv2bgr(SrcPlanes s, int w, int h, uint8_t *__restrict__ dst, int dstride)
{
    int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
    if (x >= w || y >= h) return;
    int c3[3];
    yuv_pixel(s, yuv_chroma<FMT>(s, x, y), x, y, c3);
    uint8_t *d = dst + (size_t)y * dstride + 3 * x;
    d[0] = (uint8_t)c3[0]; d[1] = (uint8_t)c3[1]; d[2] = (uint8_t)c3[2];
}

__global__ void __launch_bounds__(256)
k_bgr2gray(const uint8_t *__restrict__ src, int w, int h, int sstride, int cn, uint8_t *__restrict__ dst, int dstride)
{
    int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
    if (x >= w || y >= h) return;
    const uint8_t *p = src + (size_t)y * sstride + x * cn;
    dst[(size_t)y * dstride + x] = (uint8_t)gray_of(p[0], p[1], p[2]);
}

// Generic cv::resize(INTER_LINEAR) for cn interleaved channels; one thread per output pixel.
__global__ void __launch_bounds__(256)
k_resize_linear(const uint8_t *__restrict__ src, int sw, int sh, int sstride, int cn, uint8_t *__restrict__ dst, int dw,
                int dh, int dstride, const int *__restrict__ rtab)
{
    int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
    if (x >= dw || y >= dh) return;
    int mode = rtab[0];
    uint8_t *d = dst + (size_t)y * dstride + x * cn;
    if (mode == RT_COPY) {
        const uint8_t *p = src + (size_t)y * sstride + x * cn;
        for (int c = 0; c < cn; c++) d[c] = p[c];
    } else if (mode == RT_BOX2) {
        const uint8_t *p0 = src + (size_t)(2 * y) * sstride + 2 * x * cn, *p1 = p0 + sstride;
        for (int c = 0; c < cn; c++) d[c] = (uint8_t)((p0[c] + p0[c + cn] + p1[c] + p1[c + cn] + 2) >> 2);
    } else {
        const int *xofs = rtab + 1, *xa = xofs + dw, *y0t = xa + dw, *y1t = y0t + dh, *ybt = y1t + dh;
        int sx = xofs[x], sx1 = min(sx + 1, sw - 1), xav = xa[x], ybv = ybt[y];
        int a0 = (short)(xav & 0xFFFF), a1 = xav >> 16, b0 = (short)(ybv & 0xFFFF), b1 = ybv >> 16;
        const uint8_t *r0 = src + (size_t)y0t[y] * sstride, *r1 = src + (size_t)y1t[y] * sstride;
        for (int c = 0; c < cn; c++) d[c] = (uint8_t)lin_tap(r0, r1, sx * cn + c, sx1 * cn + c, a0, a1, b0, b1);
    }
}

__global__ void __launch_bounds__(256)
k_hist(const uint8_t *__restrict__ src, int w, int h, int stride, int *__restrict__ hist, uint8_t *__restrict__ lut)
{
    __shared__ int sh_hist[256];
    int tid = threadIdx.y * 32 + threadIdx.x;
    sh_hist[tid] = 0;
    __syncthreads();
    int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
    if (x < w && y < h) atomicAdd(&sh_hist[src[(size_t)y * stride + x]], 1);
    prep_finish(tid, sh_hist, hist, lut, w * h);                 // lut: the last block turns the histogram into the LUT (no launch of its own for the LUT)
}

__global__ void __launch_bounds__(256)
k_apply_lut(const uint8_t *__restrict__ src, int w, int h, int sstride, const uint8_t *__restrict__ lut,
            uint8_t *__restrict__ dst, int dstride)
{
    __shared__ uint8_t s_lut[256];
    s_lut[threadIdx.y * 32 + threadIdx.x] = lut[threadIdx.y * 32 + threadIdx.x];
    __syncthreads();
    int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
    if (x < w && y < h) dst[(size_t)y * dstride + x] = s_lut[src[(size_t)y * sstride + x]];
}

__global__ void __launch_bounds__(256)
k_flip(const uint8_t *__restrict__ src, int w, int h, int sstride, uint8_t *__restrict__ dst, int dstride)
{
    int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
    if (x < w && y < h) dst[(size_t)y * dstride + x] = src[(size_t)y * sstride + (w - 1 - x)];
}

// ------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------
static inline dim3 grid2d(int w, int h) { return dim3((w + 31) / 32, (h + 7) / 8); }

// persistent grids for the prep kernels: a few blocks per SM, every block flushes its histogram once
static inline int prep_grid(int tiles)
{
    if (tiles <= 148 * 6) return tiles > 0 ? tiles : 1;
    int per_block = (tiles + 148 * 6 - 1) / (148 * 6);          // every block the same number of tiles (+-1)
    return (tiles + per_block - 1) / per_block;
}
static inline bool aligned4(const void *p, int stride) { return (((uintptr_t)p | (uintptr_t)(unsigned)stride) & 3u) == 0; }

cudaError_t launch_face_prep(const uint8_t *src, int sw, int sh, int sstride, int cn, uint8_t *gray, int dw, int dh,
                             const int *rtab, int *hist, cudaStream_t st, uint8_t *lut)
{
    const int mode = (sw == dw && sh == dh) ? RT_COPY : (sw == 2 * dw && sh == 2 * dh) ? RT_BOX2 : RT_LINEAR;   // = rtab[0]
    if (mode != RT_LINEAR && cn == 3 && (dw & 3) == 0 && aligned4(src, sstride) && aligned4(gray, 0)) {
        int tiles = ((dw / 4 + 31) / 32) * ((dh + 7) / 8);
        if (mode == RT_COPY) k_face_prep_bgr4<RT_COPY, false><<<prep_grid(tiles), dim3(32, 8), 0, st>>>(src, sstride, gray, dw, dh, hist, lut);
        else k_face_prep_bgr4<RT_BOX2, false><<<prep_grid(tiles), dim3(32, 8), 0, st>>>(src, sstride, gray, dw, dh, hist, lut);
        return cudaGetLastError();
    }
    int tiles = ((dw + 31) / 32) * ((dh + 7) / 8);
    k_face_prep<false><<<prep_grid(tiles), dim3(32, 8), 0, st>>>(src, sw, sh, sstride, cn, gray, dw, dh, rtab, hist, lut);
    return cudaGetLastError();
}

cudaError_t launch_face_prep_batch(const uint8_t *const *srcs, int n, bool aligned, int sw, int sh, int sstride, uint8_t *gray,
                                   int dw, int dh, const int *rtab, int *hist, uint8_t *lut, cudaStream_t st)
{
    const int mode = (sw == dw && sh == dh) ? RT_COPY : (sw == 2 * dw && sh == 2 * dh) ? RT_BOX2 : RT_LINEAR;   // = rtab[0]
    const size_t gs = (size_t)dw * dh;
    if (mode != RT_LINEAR && (dw & 3) == 0 && aligned) {
        const dim3 grid(prep_grid(((dw / 4 + 31) / 32) * ((dh + 7) / 8)), n);
        if (mode == RT_COPY) k_face_prep_bgr4<RT_COPY, true><<<grid, dim3(32, 8), 0, st>>>(nullptr, sstride, gray, dw, dh, hist, lut, srcs, gs);
        else k_face_prep_bgr4<RT_BOX2, true><<<grid, dim3(32, 8), 0, st>>>(nullptr, sstride, gray, dw, dh, hist, lut, srcs, gs);
        return cudaGetLastError();
    }
    const dim3 grid(prep_grid(((dw + 31) / 32) * ((dh + 7) / 8)), n);
    k_face_prep<true><<<grid, dim3(32, 8), 0, st>>>(nullptr, sw, sh, sstride, 3, gray, dw, dh, rtab, hist, lut, srcs, gs);
    return cudaGetLastError();
}
template <int FMT>
static cudaError_t launch_prep_yuv_fmt(const SrcPlanes &s, int sw, int sh, uint8_t *gray, int dw, int dh, const int *rtab, int *hist,
                                       cudaStream_t st, uint8_t *lut)
{
    const int mode = (sw == dw && sh == dh) ? RT_COPY : (sw == 2 * dw && sh == 2 * dh) ? RT_BOX2 : RT_LINEAR;   // = rtab[0]
    const bool al = aligned4(s.p0, s.s0) && aligned4(s.p1, s.s1) && (FMT != 1 || aligned4(s.p2, s.s2)) && aligned4(gray, 0);
    if (mode != RT_LINEAR && (dw & 3) == 0 && al) {
        int tiles = ((dw / 4 + 31) / 32) * ((dh + 7) / 8);
        if (mode == RT_COPY) k_face_prep_yuv4<FMT, RT_COPY, false><<<prep_grid(tiles), dim3(32, 8), 0, st>>>(s, gray, dw, dh, hist, lut);
        else k_face_prep_yuv4<FMT, RT_BOX2, false><<<prep_grid(tiles), dim3(32, 8), 0, st>>>(s, gray, dw, dh, hist, lut);
        return cudaGetLastError();
    }
    int tiles = ((dw + 31) / 32) * ((dh + 7) / 8);
    k_face_prep_yuv<FMT, false><<<prep_grid(tiles), dim3(32, 8), 0, st>>>(s, sw, sh, gray, dw, dh, rtab, hist, lut);
    return cudaGetLastError();
}

// aligned: every plane pointer of every image and every plane stride is 4-byte aligned (the vectorised kernel's rule)
template <int FMT>
static cudaError_t launch_prep_yuv_batch_fmt(const uint8_t *const *planes, int n, bool aligned, const SrcPlanes &s, int sw, int sh,
                                             uint8_t *gray, int dw, int dh, const int *rtab, int *hist, uint8_t *lut, cudaStream_t st)
{
    const int mode = (sw == dw && sh == dh) ? RT_COPY : (sw == 2 * dw && sh == 2 * dh) ? RT_BOX2 : RT_LINEAR;   // = rtab[0]
    const size_t gs = (size_t)dw * dh;
    if (mode != RT_LINEAR && (dw & 3) == 0 && aligned) {
        const dim3 grid(prep_grid(((dw / 4 + 31) / 32) * ((dh + 7) / 8)), n);
        if (mode == RT_COPY) k_face_prep_yuv4<FMT, RT_COPY, true><<<grid, dim3(32, 8), 0, st>>>(s, gray, dw, dh, hist, lut, planes, gs);
        else k_face_prep_yuv4<FMT, RT_BOX2, true><<<grid, dim3(32, 8), 0, st>>>(s, gray, dw, dh, hist, lut, planes, gs);
        return cudaGetLastError();
    }
    const dim3 grid(prep_grid(((dw + 31) / 32) * ((dh + 7) / 8)), n);
    k_face_prep_yuv<FMT, true><<<grid, dim3(32, 8), 0, st>>>(s, sw, sh, gray, dw, dh, rtab, hist, lut, planes, gs);
    return cudaGetLastError();
}

cudaError_t launch_face_prep_yuv_batch(int fmt, const uint8_t *const *planes, int n, bool aligned, int s0, int s1, int s2, int sw,
                                       int sh, uint8_t *gray, int dw, int dh, const int *rtab, int *hist, uint8_t *lut, cudaStream_t st)
{
    const SrcPlanes s = {nullptr, nullptr, nullptr, s0, s1, s2};
    if (fmt == NV_FMT_I420) return launch_prep_yuv_batch_fmt<1>(planes, n, aligned, s, sw, sh, gray, dw, dh, rtab, hist, lut, st);
    if (fmt == NV_FMT_NV12) return launch_prep_yuv_batch_fmt<2>(planes, n, aligned, s, sw, sh, gray, dw, dh, rtab, hist, lut, st);
    if (fmt == NV_FMT_NV21) return launch_prep_yuv_batch_fmt<3>(planes, n, aligned, s, sw, sh, gray, dw, dh, rtab, hist, lut, st);
    return cudaErrorInvalidValue;
}

cudaError_t launch_face_prep_yuv(int fmt, const SrcPlanes &s, int sw, int sh, uint8_t *gray, int dw, int dh, const int *rtab,
                                 int *hist, cudaStream_t st, uint8_t *lut)
{
    if (fmt == NV_FMT_I420) return launch_prep_yuv_fmt<1>(s, sw, sh, gray, dw, dh, rtab, hist, st, lut);
    if (fmt == NV_FMT_NV12) return launch_prep_yuv_fmt<2>(s, sw, sh, gray, dw, dh, rtab, hist, st, lut);
    if (fmt == NV_FMT_NV21) return launch_prep_yuv_fmt<3>(s, sw, sh, gray, dw, dh, rtab, hist, st, lut);
    return cudaErrorInvalidValue;
}
cudaError_t launch_yuv2gray(int fmt, const SrcPlanes &s, int w, int h, uint8_t *dst, int dstride, cudaStream_t st)
{
    dim3 g = grid2d(w, h), b(32, 8);
    if (fmt == NV_FMT_I420) k_yuv2gray<1><<<g, b, 0, st>>>(s, w, h, dst, dstride);
    else if (fmt == NV_FMT_NV12) k_yuv2gray<2><<<g, b, 0, st>>>(s, w, h, dst, dstride);
    else if (fmt == NV_FMT_NV21) k_yuv2gray<3><<<g, b, 0, st>>>(s, w, h, dst, dstride);
    else return cudaErrorInvalidValue;
    return cudaGetLastError();
}
cudaError_t launch_yuv2bgr(int fmt, const SrcPlanes &s, int w, int h, uint8_t *dst, int dstride, cudaStream_t st)
{
    dim3 g = grid2d(w, h), b(32, 8);
    if (fmt == NV_FMT_I420) k_yuv2bgr<1><<<g, b, 0, st>>>(s, w, h, dst, dstride);
    else if (fmt == NV_FMT_NV12) k_yuv2bgr<2><<<g, b, 0, st>>>(s, w, h, dst, dstride);
    else if (fmt == NV_FMT_NV21) k_yuv2bgr<3><<<g, b, 0, st>>>(s, w, h, dst, dstride);
    else return cudaErrorInvalidValue;
    return cudaGetLastError();
}
cudaError_t launch_bgr2gray(const uint8_t *src, int w, int h, int sstride, int cn, uint8_t *dst, int dstride,
                            cudaStream_t st)
{
    k_bgr2gray<<<grid2d(w, h), dim3(32, 8), 0, st>>>(src, w, h, sstride, cn, dst, dstride);
    return cudaGetLastError();
}
cudaError_t launch_resize_linear(const uint8_t *src, int sw, int sh, int sstride, int cn, uint8_t *dst, int dw, int dh,
                                 int dstride, const int *rtab, cudaStream_t st)
{
    k_resize_linear<<<grid2d(dw, dh), dim3(32, 8), 0, st>>>(src, sw, sh, sstride, cn, dst, dw, dh, dstride, rtab);
    return cudaGetLastError();
}
cudaError_t launch_hist(const uint8_t *src, int w, int h, int stride, int *hist, cudaStream_t st, uint8_t *lut)
{
    k_hist<<<grid2d(w, h), dim3(32, 8), 0, st>>>(src, w, h, stride, hist, lut);
    return cudaGetLastError();
}
cudaError_t launch_apply_lut(const uint8_t *src, int w, int h, int sstride, const uint8_t *lut, uint8_t *dst, int dstride,
                             cudaStream_t st)
{
    k_apply_lut<<<grid2d(w, h), dim3(32, 8), 0, st>>>(src, w, h, sstride, lut, dst, dstride);
    return cudaGetLastError();
}
cudaError_t launch_flip(const uint8_t *src, int w, int h, int sstride, uint8_t *dst, int dstride, cudaStream_t st)
{
    k_flip<<<grid2d(w, h), dim3(32, 8), 0, st>>>(src, w, h, sstride, dst, dstride);
    return cudaGetLastError();
}
