// kernels_pyramid.cu — K4 + K5: the cascade's internal scale pyramid (INTER_LINEAR_EXACT, always from the
// equalised base image; SURVEY.md A.4) fused with the row pass of the integral / squared-integral images
// (A.5), then the column pass.  All levels of a frame go through ONE launch of each kernel.
//
// Integral layout (chosen for the consumer, the cascade kernels): per level an (lh+1) x (lw+1) image of
// uint32 (sum is int32 in OpenCV; both are consumed through differences, so modulo-2^32 arithmetic on
// uint32 is bit-identical).  For ystep==2 levels the columns of every row are de-interleaved into an
// even plane and an odd plane (physical col = (c % ystep) * iplane + c / ystep): the cascade only visits
// even x there, so the 32 lanes of a warp, on windows x, x+2, x+4 …, read CONSECUTIVE words for every
// feature corner (coalesced in global memory, conflict-free once staged in shared memory).
#include "internal.h"

__device__ __forceinline__ int find_level(const PlanDev *__restrict__ plan, int idx, int LevelDesc::*first)
{
    int n = plan->nlevels, l = 0;
    while (l + 1 < n && plan->lv[l + 1].*first <= idx) l++;
    return l;
}

// One warp per level row, FOUR integral columns per lane and iteration (columns c0 + 4 * lane + k, i.e. pixels
// x = c - 1; column 0 is the zero column, pixel -1 counts 0): resize (two source rows, two source columns, 8.8 x 8.8
// fixed point, coefficient tables without special cases — see exact_coefs) -> equalised value -> running sums of v and
// v * v inside the lane, ONE warp-shuffle scan of the lane totals per 128 columns, a 16-byte store per array (two
// 8-byte stores on the de-interleaved ystep-2 layout: columns c, c + 2 are neighbours in the even plane, c + 1, c + 3
// in the odd one).  Round 1's kernel did one pixel per lane: 3.4 x the instructions, and a 1920-pixel row was a chain
// of 60 dependent load -> scan -> carry rounds where this one has 15.
// BATCH: image blockIdx.y reads grays[blockIdx.y] through the LUT at blockIdx.y * lut_stride and writes the integrals at
// blockIdx.y * integ_stride elements.
template <bool BATCH>
// 32 registers, no spills: eight blocks per SM (40.3 -> 38.9 us alone); the batched form needs 40 (six blocks per SM) not to spill
__global__ void __launch_bounds__(256, BATCH ? 6 : 8)
k_pyr_rowscan(const PlanDev *__restrict__ plan, const uint8_t *__restrict__ gray, int gstride,
              const uint8_t *__restrict__ lut, const int2 *__restrict__ ptab, uint32_t *__restrict__ sum,
              uint32_t *__restrict__ sq, uint8_t *__restrict__ pyr_debug, const uint8_t *const *__restrict__ grays = nullptr,
              int lut_stride = 0, unsigned integ_stride = 0)
{
    __shared__ uint8_t s_lut[256];
    int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (BATCH) lut += blockIdx.y * lut_stride;
    s_lut[tid] = lut[tid];
    __syncthreads();

    int l = find_level(plan, blockIdx.x, &LevelDesc::rowblk0);
    const LevelDesc &L = plan->lv[l];
    const int lw = L.lw, lh = L.lh, ys = L.ystep, pitch = L.ipitch, plane = L.iplane;
    int y = (blockIdx.x - L.rowblk0) * 8 + warp;
    if (y >= lh) return;
    const size_t iofs = L.iofs + (BATCH ? (size_t)blockIdx.y * integ_stride : 0);
    uint32_t *srow = sum + iofs, *qrow = sq + iofs;
    if (y == 0)                                         // first integral row is all zeros (pitch is a multiple of 4)
        for (int c = lane * 4; c < pitch; c += 128) {
            *reinterpret_cast<uint4 *>(srow + c) = make_uint4(0, 0, 0, 0);
            *reinterpret_cast<uint4 *>(qrow + c) = make_uint4(0, 0, 0, 0);
        }
    srow += (size_t)(y + 1) * pitch;
    qrow += (size_t)(y + 1) * pitch;

    const int4 *xt = reinterpret_cast<const int4 *>(ptab + L.xtab);     // two (index, fraction) entries per int4
    int2 ty = (ptab + L.ytab)[y];
    if (BATCH) gray = grays[blockIdx.y];
    const uint8_t *g0 = gray + (size_t)ty.x * gstride, *g1 = g0 + gstride;
    const uint32_t r1 = (uint32_t)ty.y, r0 = 256u - r1;
    uint32_t carry_s = 0, carry_q = 0;
    for (int c0 = 0; c0 <= lw; c0 += 128) {
        const int c = c0 + lane * 4;
        uint32_t v[4] = {0, 0, 0, 0};
        if (c <= lw) {
            int4 ta = xt[c >> 1], tb = xt[(c >> 1) + 1];
            const int ix[4] = {ta.x, ta.z, tb.x, tb.z};
            const uint32_t fx[4] = {(uint32_t)ta.y, (uint32_t)ta.w, (uint32_t)tb.y, (uint32_t)tb.w};
#pragma unroll
            for (int k = 0; k < 4; k++) {
                uint32_t c1 = fx[k], cz = 256u - c1;
                uint32_t h0 = s_lut[g0[ix[k]]] * cz + s_lut[g0[ix[k] + 1]] * c1;
                uint32_t h1 = s_lut[g1[ix[k]]] * cz + s_lut[g1[ix[k] + 1]] * c1;
                uint32_t val = (h0 * r0 + h1 * r1 + 32768u) >> 16;
                int x = c + k - 1;
                v[k] = (unsigned)x < (unsigned)lw ? val : 0u;           // pixel -1 (column 0) and the padding columns count 0
            }
            if (pyr_debug) {
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    int x = c + k - 1;
                    if ((unsigned)x < (unsigned)lw) pyr_debug[L.pofs + (size_t)y * lw + x] = (uint8_t)v[k];
                }
            }
        }
        uint32_t s0 = v[0], s1 = s0 + v[1], s2 = s1 + v[2], s3 = s2 + v[3];
        uint32_t q0 = v[0] * v[0], q1 = v[1] * v[1] + q0, q2 = v[2] * v[2] + q1, q3 = v[3] * v[3] + q2;
        uint32_t s = s3, q = q3;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            uint32_t ts = __shfl_up_sync(0xffffffffu, s, d), tq = __shfl_up_sync(0xffffffffu, q, d);
            if (lane >= d) { s += ts; q += tq; }
        }
        s += carry_s; q += carry_q;                     // inclusive through this lane's four columns
        const uint32_t bs = s - s3, bq = q - q3;
        if (c <= lw) {                                  // the lane's four columns exist together (pitch / plane are multiples of 4)
            if (ys == 2) {
                const int pc = c >> 1;
                *reinterpret_cast<uint2 *>(srow + pc) = make_uint2(bs + s0, bs + s2);
                *reinterpret_cast<uint2 *>(srow + plane + pc) = make_uint2(bs + s1, s);
                *reinterpret_cast<uint2 *>(qrow + pc) = make_uint2(bq + q0, bq + q2);
                *reinterpret_cast<uint2 *>(qrow + plane + pc) = make_uint2(bq + q1, q);
            } else {
                *reinterpret_cast<uint4 *>(srow + c) = make_uint4(bs + s0, bs + s1, bs + s2, s);
                *reinterpret_cast<uint4 *>(qrow + c) = make_uint4(bq + q0, bq + q1, bq + q2, q);
            }
        }
        carry_s = __shfl_sync(0xffffffffu, s, 31);
        carry_q = __shfl_sync(0xffffffffu, q, 31);
    }
}

// Column pass, shared-memory tiled: a block owns NV_COLBLK = 128 physical columns of one array of one level (four per
// lane, moved as 16-byte vectors); its 16 warps split the rows into 16 bands.  Pass 1 sums each band, the band totals
// are exchanged through shared memory and prefixed, pass 2 re-reads the band (L1/L2 hit) and writes the running
// column sums.  Every global access is a 512-byte row segment.
__device__ __forceinline__ uint4 add4(uint4 a, uint4 b) { return make_uint4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }

// 16 bands = 512 threads x 40 registers, 8 KB of shared memory: small enough to share an SM with resident blocks of the
// cascade kernel of another stream.  With 32 bands (1024 threads, a whole SM's worth of registers) the column scan had
// to wait for an SM to drain: bench.py 2418 -> 2536 frames/s from this change alone (profiles/r1_v5_summary.md).
#ifndef NV_COLBANDS
#define NV_COLBANDS 16
#endif
template <bool BATCH>                                             // BATCH: image blockIdx.y, integrals at blockIdx.y * integ_stride
__global__ void __launch_bounds__(32 * NV_COLBANDS, BATCH ? 2 : 0)   // the batched form spills at the 40 registers ptxas picks unbounded
k_colscan(const PlanDev *__restrict__ plan, int total_colblk, uint32_t *__restrict__ sum, uint32_t *__restrict__ sq,
          unsigned integ_stride = 0)
{
    __shared__ uint4 tot[NV_COLBANDS][33];
    int lane = threadIdx.x & 31, band = threadIdx.x >> 5;
    int b = blockIdx.x;
    uint32_t *arr = sum;
    if (b >= total_colblk) { b -= total_colblk; arr = sq; }
    if (BATCH) arr += (size_t)blockIdx.y * integ_stride;
    int l = find_level(plan, b, &LevelDesc::colblk0);
    const LevelDesc &L = plan->lv[l];
    const int pitch = L.ipitch, rows = L.lh + 1;
    int col = (b - L.colblk0) * NV_COLBLK + lane * 4;
    bool ok = col < pitch;                              // pitch is a multiple of 4: a lane's four columns exist together
    uint4 *p = reinterpret_cast<uint4 *>(arr + L.iofs + col);
    const size_t rs = (size_t)(pitch >> 2);             // row stride in uint4
    int R = (rows + NV_COLBANDS - 1) / NV_COLBANDS, r0 = band * R, r1 = min(rows, r0 + R);
    uint4 acc = make_uint4(0, 0, 0, 0);
    if (ok) {
        const uint4 *q = p + (size_t)r0 * rs;
        int r = r0;
        for (; r + 4 <= r1; r += 4, q += 4 * rs) {
            uint4 a0 = q[0], a1 = q[rs], a2 = q[2 * rs], a3 = q[3 * rs];
            acc = add4(acc, add4(add4(a0, a1), add4(a2, a3)));
        }
        for (; r < r1; r++, q += rs) acc = add4(acc, q[0]);
    }
    tot[band][lane] = acc;
    __syncthreads();
    uint4 run = make_uint4(0, 0, 0, 0);
    for (int k = 0; k < band; k++) run = add4(run, tot[k][lane]);
    if (ok) {
        uint4 *q = p + (size_t)r0 * rs;
        int r = r0;
        for (; r + 4 <= r1; r += 4, q += 4 * rs) {
            uint4 a0 = q[0], a1 = q[rs], a2 = q[2 * rs], a3 = q[3 * rs];
            a0 = add4(a0, run); a1 = add4(a1, a0); a2 = add4(a2, a1); a3 = add4(a3, a2);
            q[0] = a0; q[rs] = a1; q[2 * rs] = a2; q[3 * rs] = a3;
            run = a3;
        }
        for (; r < r1; r++, q += rs) { run = add4(run, q[0]); q[0] = run; }
    }
}

// Tilted integral (cv::integral's third output; only for cascades with tilted features).  tilted(X,Y) = sum of the
// level's pixels in the 45-degree triangle whose apex is pixel (X-1, Y-1).  Row y < Y of the triangle is the pixel run
// [X-1-k, X-1+k], k = Y-1-y, clipped to the image, i.e. R(y, cl(X+k)) - R(y, cl(X-1-k)) with the row prefix
// R(y, x) = sum[y+1][x] - sum[y][x] taken from the finished upright integral and cl() clamping to [0, lw].  So
//   tilted(X,Y) = A(X,Y) - B(X,Y),   A = sum_y R(y, cl(X+Y-1-y)),   B = sum_y R(y, cl(X-Y+y)),
// and A only depends on the anti-diagonal d = X+Y, B on the diagonal e = X-Y: ONE THREAD PER DIAGONAL walks down its
// diagonal keeping a running sum (a thread's leading rows, where the run is clipped to a whole row or to nothing,
// collapse to sum[y0][lw] or 0), no synchronisation, consecutive threads on consecutive addresses.  Pass A writes,
// pass B subtracts.  Plain row layout, pitch and level offsets shared with the upright integrals.
struct TiltView {
    const uint32_t *S; uint32_t *T; int lw, lh, pitch, plane, ys;
    __device__ __forceinline__ uint32_t s(int y, int x) const { return __ldg(S + (size_t)y * pitch + (ys == 2 ? (x & 1) * plane + (x >> 1) : x)); }
};

__device__ __forceinline__ bool tilt_setup(const PlanDev *__restrict__ plan, const uint32_t *sum, uint32_t *tilt, TiltView &v, int &i)
{
    int l = find_level(plan, blockIdx.x, &LevelDesc::dblk0);
    const LevelDesc &L = plan->lv[l];
    v = TiltView{sum + L.iofs, tilt + L.iofs, L.lw, L.lh, L.ipitch, L.iplane, L.ystep};
    i = (blockIdx.x - L.dblk0) * 256 + threadIdx.x;              // diagonal index, 0 .. lw + lh - 1
    return i < L.lw + L.lh;
}

__global__ void __launch_bounds__(256)
k_tilt_a(const PlanDev *__restrict__ plan, const uint32_t *__restrict__ sum, uint32_t *__restrict__ tilt)
{
    TiltView v; int i;
    if (!tilt_setup(plan, sum, tilt, v, i)) return;
    const int d = i + 1;                                         // X + Y, 1 .. lw + lh
    if (d - 1 <= v.lw) v.T[d - 1] = 0u;                          // row Y = 0
    int y0 = max(0, d - 1 - v.lw);                               // rows above y0: the run is clipped to the whole row
    uint32_t acc = v.s(y0, v.lw);
    for (int y = y0; y < v.lh && y < d; y++) {
        int X = d - 1 - y;                                       // 0 <= X <= lw here
        acc += v.s(y + 1, X) - v.s(y, X);
        v.T[(size_t)(y + 1) * v.pitch + X] = acc;
    }
}

__global__ void __launch_bounds__(256)
k_tilt_b(const PlanDev *__restrict__ plan, const uint32_t *__restrict__ sum, uint32_t *__restrict__ tilt)
{
    TiltView v; int i;
    if (!tilt_setup(plan, sum, tilt, v, i)) return;
    const int e = i - v.lh;                                      // X - Y, -lh .. lw - 1
    uint32_t acc = 0u;
    for (int y = max(0, -e); y < v.lh; y++) {                    // rows above: the run starts left of the image
        int X = e + y + 1;
        if (X > v.lw) break;
        acc += v.s(y + 1, X - 1) - v.s(y, X - 1);                // R(y, X - 1), 0 <= X - 1 < lw
        v.T[(size_t)(y + 1) * v.pitch + X] -= acc;
    }
}

cudaError_t launch_tilted(const PlanDev *plan, int total_dblk, const uint32_t *sum, uint32_t *tilt, cudaStream_t st)
{
    k_tilt_a<<<total_dblk, 256, 0, st>>>(plan, sum, tilt);
    k_tilt_b<<<total_dblk, 256, 0, st>>>(plan, sum, tilt);
    return cudaGetLastError();
}

cudaError_t launch_pyr_rowscan(const PlanDev *plan, int total_rowblk, const uint8_t *gray, int gstride, const uint8_t *lut,
                               const int *ptab, uint32_t *sum, uint32_t *sq, uint8_t *pyr_debug, cudaStream_t st)
{
    k_pyr_rowscan<false><<<total_rowblk, 256, 0, st>>>(plan, gray, gstride, lut, (const int2 *)ptab, sum, sq, pyr_debug);
    return cudaGetLastError();
}

cudaError_t launch_colscan(const PlanDev *plan, int total_colblk, uint32_t *sum, uint32_t *sq, cudaStream_t st)
{
    k_colscan<false><<<2 * total_colblk, 32 * NV_COLBANDS, 0, st>>>(plan, total_colblk, sum, sq);
    return cudaGetLastError();
}

cudaError_t launch_pyramid_batch(const PlanDev *plan, int total_rowblk, int total_colblk, int n, const uint8_t *const *grays, int gstride,
                                 const uint8_t *lut, int lut_stride, const int *ptab, uint32_t *sum, uint32_t *sq, size_t integ_stride,
                                 cudaStream_t st)
{
    k_pyr_rowscan<true><<<dim3(total_rowblk, n), 256, 0, st>>>(plan, nullptr, gstride, lut, (const int2 *)ptab, sum, sq, nullptr, grays,
                                                               lut_stride, (unsigned)integ_stride);
    k_colscan<true><<<dim3(2 * total_colblk, n), 32 * NV_COLBANDS, 0, st>>>(plan, total_colblk, sum, sq, (unsigned)integ_stride);
    return cudaGetLastError();
}
