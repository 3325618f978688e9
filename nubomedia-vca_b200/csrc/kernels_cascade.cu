// kernels_cascade.cu — K6 + K7: Haar cascade stage evaluation over every level of the pyramid.
// Replaces the inside of cv::CascadeClassifier::detectMultiScale (kmsfacedetect.cpp:809-811 and the
// analogous calls of the eye/mouth/nose/ear elements).  Arithmetic per SURVEY.md A.6 plus the three
// facts the oracle probes added (oracle/nubo_oracle.c): leaves accumulate in DOUBLE, the stage
// threshold is (float)xml - 1e-5f, a window is valid iff area * (float)(1/sqrt(nf)) < 0.1.
// No FMA contraction anywhere on the float path: explicit __fmul_rn / __fadd_rn.
//
// The pass structure is described above k_stage0_rows.  k_alive_to_queue + k_queue_stages (one thread per alive
// window, plain early-exit loop) is the generic path for cascades the tile kernel cannot take (window wider or
// taller than 32); k_stage0_rows is the generic form of k_stage0_rows_p (more than 8 stage-0 classifiers).
#include "cascade_eval.cuh"

#include <set>

__device__ __forceinline__ int find_level_c(const PlanDev *__restrict__ plan, int idx, int LevelDesc::*first)
{
    int n = plan->nlevels, l = 0;
    while (l + 1 < n && plan->lv[l + 1].*first <= idx) l++;
    return l;
}

// warp-uniform warp index, rebuilt from votes so that the compiler can prove it (see uniformize below)
__device__ __forceinline__ int uniformize_s0(int v)
{
    int r = 0;
    for (int k = 0; k < 3; k++) r |= (int)(__ballot_sync(0xffffffffu, (v >> k) & 1) & (1u << k));
    return r;
}

// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_queue_stages(const PlanDev *__restrict__ plan, const DevCascade *__restrict__ meta, const DevStump *__restrict__ stumps,
               const uint32_t *__restrict__ sum, const uint2 *__restrict__ queue, int *__restrict__ counters,
               uint32_t *__restrict__ cand, int cand_cap, int16_t *__restrict__ depth)
{
    int n = counters[0];
    int nstages = meta->nstages;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        uint2 q = queue[i];
        int l = q.x >> 26, iy = (q.x >> 13) & 8191, ix = q.x & 8191;
        float vnf = __uint_as_float(q.y);
        const LevelDesc &L = plan->lv[l];
        LevelView v{sum + L.iofs, L.ipitch, L.iplane, L.ystep};
        const uint32_t *wb = v.sum + (size_t)iy * L.ystep * L.ipitch + ix;
        int code = NV_DEPTH_PASS;
        for (int st = 1; st < nstages; st++) {
            double tmp = 0.;
            int s0 = meta->stage_first[st], s1 = meta->stage_first[st + 1];
            for (int k = s0; k < s1; k++) {
                StumpRegs s = load_stump(stumps + k);
                tmp = __dadd_rn(tmp, (double)stump_leaf(wb, v, s, vnf));
            }
            if (tmp < (double)meta->stage_thr[st]) { code = -st; break; }
        }
        if (depth) depth[L.wofs + iy * L.nx + ix] = (int16_t)code;
        if (code == NV_DEPTH_PASS) {
            int pos = atomicAdd(&counters[1], 1);
            if (pos < cand_cap) cand[pos] = q.x;
            else counters[2] = 1;
        }
    }
}

// ================================================================================================
// General cascades (OpenCV's predictOrdered path): weak classifiers that are trees of more than one node and/or
// features on the tilted integral.  One thread per window, plain early-exit loops; these models run in the nested
// ROI stages of the eye / mouth / nose / ear elements, where a call has 10^3..10^4 windows.
// ================================================================================================
__device__ __forceinline__ uint32_t skip_rule_word(uint32_t f, bool &e);

__global__ void __launch_bounds__(256)
k_stage0_rows_gen(const PlanDev *__restrict__ plan, int total_rows, const DevCascade *__restrict__ meta, const GenModel g,
                  const uint32_t *__restrict__ sum, const uint32_t *__restrict__ sq, const uint32_t *__restrict__ tilt,
                  float *__restrict__ vnf_out, uint32_t *__restrict__ bits_alive, int *__restrict__ counters,
                  int16_t *__restrict__ depth)
{
    int lane = threadIdx.x & 31;
    int row = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= total_rows) return;
    int l = find_level_c(plan, row, &LevelDesc::row0);
    const LevelDesc &L = plan->lv[l];
    int iy = row - L.row0;
    LevelView v{sum + L.iofs, L.ipitch, L.iplane, L.ystep};
    int ww = plan->win_w, wh = plan->win_h;
    int c00 = corner(v, 1, 1), c10 = corner(v, ww - 1, 1), c01 = corner(v, 1, wh - 1), c11 = corner(v, ww - 1, wh - 1);
    double area = (double)((ww - 2) * (wh - 2));
    int n0 = meta->stage_first[1];
    double thr0 = (double)meta->stage_thr[0];
    size_t rowbase = (size_t)iy * L.ystep * L.ipitch;
    bool e = true;
    int nalive = 0;
    for (int cx = 0; cx < L.nxw; cx++) {
        int ix = cx * 32 + lane;
        bool valid = ix < L.nx;
        int ixc = valid ? ix : L.nx - 1;
        const uint32_t *wb = v.sum + rowbase + ixc, *qb = sq + L.iofs + rowbase + ixc;
        const uint32_t *tb = tilt ? tilt + L.iofs + rowbase + ixc * L.ystep : nullptr;
        float vnf = 0.f;
        bool ok = g.subset != nullptr;                            // LBP: no variance normalisation, every window is evaluated
        if (!ok) {
            int valsum = (int)(__ldg(wb + c00) - __ldg(wb + c10) - __ldg(wb + c01) + __ldg(wb + c11));
            uint32_t valsq = __ldg(qb + c00) - __ldg(qb + c10) - __ldg(qb + c01) + __ldg(qb + c11);
            double nf = __dsub_rn(__dmul_rn(area, (double)valsq), __dmul_rn((double)valsum, (double)valsum));
            if (nf > 0.) {
                vnf = __double2float_rn(__ddiv_rn(1.0, __dsqrt_rn(nf)));
                ok = __dmul_rn(area, (double)vnf) < 1e-1;
            }
        }
        bool fail = false;
        if (ok) fail = gen_stage_sum(g, 0, n0, wb, v, tb, L.ipitch, vnf) < thr0;
        ok = ok && valid;
        fail = fail && ok;
        uint32_t f = __ballot_sync(0xffffffffu, fail);
        uint32_t em = skip_rule_word(f, e);
        bool visited = (em >> lane) & 1u;
        bool alive = visited && ok && !fail;
        uint32_t am = __ballot_sync(0xffffffffu, alive);
        nalive += __popc(am);
        if (lane == 0) bits_alive[L.bofs + iy * L.nxw + cx] = am;
        if (alive) vnf_out[L.wofs + iy * L.nx + ix] = vnf;
        if (depth && valid && !alive)
            depth[L.wofs + iy * L.nx + ix] = (int16_t)(!visited ? NV_DEPTH_SKIPPED : (!ok ? NV_DEPTH_VARREJ : 0));
    }
    if (lane == 0 && nalive) atomicAdd(&counters[0], nalive);
}

__global__ void __launch_bounds__(256)
k_queue_stages_gen(const PlanDev *__restrict__ plan, const DevCascade *__restrict__ meta, const GenModel g,
                   const uint32_t *__restrict__ sum, const uint32_t *__restrict__ tilt, const uint2 *__restrict__ queue,
                   int *__restrict__ counters, uint32_t *__restrict__ cand, int cand_cap, int16_t *__restrict__ depth)
{
    int n = counters[0];
    int nstages = meta->nstages;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        uint2 q = queue[i];
        int l = q.x >> 26, iy = (q.x >> 13) & 8191, ix = q.x & 8191;
        float vnf = __uint_as_float(q.y);
        const LevelDesc &L = plan->lv[l];
        LevelView v{sum + L.iofs, L.ipitch, L.iplane, L.ystep};
        size_t rowbase = (size_t)iy * L.ystep * L.ipitch;
        const uint32_t *wb = v.sum + rowbase + ix;
        const uint32_t *tb = tilt ? tilt + L.iofs + rowbase + ix * L.ystep : nullptr;
        int code = NV_DEPTH_PASS;
        for (int st = 1; st < nstages; st++)
            if (gen_stage_sum(g, meta->stage_first[st], meta->stage_first[st + 1], wb, v, tb, L.ipitch, vnf) <
                (double)meta->stage_thr[st]) { code = -st; break; }
        if (depth) depth[L.wofs + iy * L.nx + ix] = (int16_t)code;
        if (code == NV_DEPTH_PASS) {
            int pos = atomicAdd(&counters[1], 1);
            if (pos < cand_cap) cand[pos] = q.x;
            else counters[2] = 1;
        }
    }
}

// The same with one WARP per window and one lane per tree of the stage (exact when the stage sums are order-free,
// cascade_xml.cpp): a window that passes twenty stages of twenty trees is twenty rounds of tree walks deep instead of
// four hundred, which is what the latency of a small nested-ROI call is made of.  Windows are handed out dynamically.
__global__ void __launch_bounds__(256)
k_queue_stages_gen_warp(const PlanDev *__restrict__ plan, const DevCascade *__restrict__ meta, const GenModel g,
                        const uint32_t *__restrict__ sum, const uint32_t *__restrict__ tilt, const uint2 *__restrict__ queue,
                        int *__restrict__ counters, uint32_t *__restrict__ cand, int cand_cap, int16_t *__restrict__ depth,
                        int stage_begin, int cin)
{
    const int lane = threadIdx.x & 31;
    const int n = counters[cin], nstages = meta->nstages;
    for (;;) {
        int e = 0;
        if (lane == 0) e = atomicAdd(&counters[5], 1);
        e = __shfl_sync(0xffffffffu, e, 0);
        if (e >= n) break;
        uint2 q = queue[e];
        int l = q.x >> 26, iy = (q.x >> 13) & 8191, ix = q.x & 8191;
        float vnf = __uint_as_float(q.y);
        const LevelDesc &L = plan->lv[l];
        LevelView v{sum + L.iofs, L.ipitch, L.iplane, L.ystep};
        size_t rowbase = (size_t)iy * L.ystep * L.ipitch;
        const uint32_t *wb = v.sum + rowbase + ix;
        const uint32_t *tb = tilt ? tilt + L.iofs + rowbase + ix * L.ystep : nullptr;
        int code = NV_DEPTH_PASS;
        for (int st = stage_begin; st < nstages; st++) {
            const int t0 = meta->stage_first[st], t1 = meta->stage_first[st + 1];
            double tmp = 0.;
            for (int t = t0 + lane; t < t1; t += 32) tmp = __dadd_rn(tmp, gen_stage_sum(g, t, t + 1, wb, v, tb, L.ipitch, vnf));
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) tmp = __dadd_rn(tmp, __shfl_xor_sync(0xffffffffu, tmp, d));
            if (tmp < (double)meta->stage_thr[st]) { code = -st; break; }
        }
        if (lane == 0) {
            if (depth) depth[L.wofs + iy * L.nx + ix] = (int16_t)code;
            if (code == NV_DEPTH_PASS) {
                int pos = atomicAdd(&counters[1], 1);
                if (pos < cand_cap) cand[pos] = q.x;
                else counters[2] = 1;
            }
        }
    }
}

// Large plans (a full frame through a tree / tilted model): one thread per queued window over the stage range
// [sb, se) only, survivors compacted into the next queue (warp-aggregated append), so that every pass starts with full
// warps again — the early stages of such a model reject nine windows in ten, and a warp per window (above) spends its
// 32 lanes on a handful of trees there.  Sums run in XML order: exact for every model, no certificate needed.
// final != 0: [sb, se) reaches the last stage and survivors are candidates.
__global__ void __launch_bounds__(256)
k_queue_range_gen(const PlanDev *__restrict__ plan, const DevCascade *__restrict__ meta, const GenModel g,
                  const uint32_t *__restrict__ sum, const uint32_t *__restrict__ tilt, const uint2 *__restrict__ qin,
                  uint2 *__restrict__ qout, int qcap, int *__restrict__ counters, int cin, int cout, uint32_t *__restrict__ cand,
                  int cand_cap, int16_t *__restrict__ depth, int sb, int se, int final)
{
    const int n = counters[cin], lane = threadIdx.x & 31;
    const int nround = (n + 31) & ~31;                            // whole warps stay in the loop: the append below votes
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nround; i += gridDim.x * blockDim.x) {
        bool pass = false;
        uint2 q = make_uint2(0u, 0u);
        if (i < n) {
            q = qin[i];
            int l = q.x >> 26, iy = (q.x >> 13) & 8191, ix = q.x & 8191;
            float vnf = __uint_as_float(q.y);
            const LevelDesc &L = plan->lv[l];
            LevelView v{sum + L.iofs, L.ipitch, L.iplane, L.ystep};
            size_t rowbase = (size_t)iy * L.ystep * L.ipitch;
            const uint32_t *wb = v.sum + rowbase + ix;
            const uint32_t *tb = tilt ? tilt + L.iofs + rowbase + ix * L.ystep : nullptr;
            int code = NV_DEPTH_PASS;
            for (int st = sb; st < se; st++)
                if (gen_stage_sum(g, meta->stage_first[st], meta->stage_first[st + 1], wb, v, tb, L.ipitch, vnf) <
                    (double)meta->stage_thr[st]) { code = -st; break; }
            pass = code == NV_DEPTH_PASS;
            if (depth && (!pass || final)) depth[L.wofs + iy * L.nx + ix] = (int16_t)code;
        }
        const unsigned m = __ballot_sync(0xffffffffu, pass);
        if (m) {
            int base = 0;
            if (lane == 0) base = atomicAdd(&counters[final ? 1 : cout], __popc(m));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (pass) {
                const int pos = base + __popc(m & ((1u << lane) - 1u));
                if (final) { if (pos < cand_cap) cand[pos] = q.x; else counters[2] = 1; }
                else { if (pos < qcap) qout[pos] = q; else counters[2] = 1; }
            }
        }
    }
}

// ================================================================================================
// pass structure (all levels per launch):
//   k_stage0_rows      one warp per window ROW: variance + stage 0 for each 32-window chunk, the skip
//                      automaton carried along the row in a register, one "alive" bit-word per chunk.
//   k_cascade_classes  one block per 64x32-window tile: the integral tile (+halo) is staged in shared
//                      memory by TMA, stages 1..B-1 run with each lane bound to one shared-memory bank
//                      class of windows (see the kernel).  The weak classifiers of these stages and the
//                      tensor maps sit in the kernel's parameter (constant) bank.
//   k_cascade_tail     the few windows that outlive the bulk stages: one warp per window, the 32 lanes
//                      evaluate 32 different weak classifiers of the stage on a private copy of the
//                      window's integral patch; exact because the double stage sum is order-free for the
//                      cascade (certificate computed at load), sequential shuffles otherwise.
// ================================================================================================
__global__ void __launch_bounds__(256)
k_stage0_rows(const PlanDev *__restrict__ plan, int total_rows, const DevCascade *__restrict__ meta,
              const DevStump *__restrict__ stumps, const uint32_t *__restrict__ sum, const uint32_t *__restrict__ sq,
              float *__restrict__ vnf_out, uint32_t *__restrict__ bits_alive, int *__restrict__ counters,
              int16_t *__restrict__ depth)
{
    int lane = threadIdx.x & 31;
    int row = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= total_rows) return;
    int l = find_level_c(plan, row, &LevelDesc::row0);
    const LevelDesc &L = plan->lv[l];
    int iy = row - L.row0;
    LevelView v{sum + L.iofs, L.ipitch, L.iplane, L.ystep};
    int ww = plan->win_w, wh = plan->win_h;
    int c00 = corner(v, 1, 1), c10 = corner(v, ww - 1, 1), c01 = corner(v, 1, wh - 1), c11 = corner(v, ww - 1, wh - 1);
    double area = (double)((ww - 2) * (wh - 2));
    int n0 = meta->stage_first[1];
    double thr0 = (double)meta->stage_thr[0];
    size_t rowbase = (size_t)iy * L.ystep * L.ipitch;
    bool e = true;                                   // is the next window visited?  (x = 0 always is)
    int nalive = 0;
    for (int cx = 0; cx < L.nxw; cx++) {
        int ix = cx * 32 + lane;
        bool valid = ix < L.nx;
        int ixc = valid ? ix : L.nx - 1;
        const uint32_t *wb = v.sum + rowbase + ixc, *qb = sq + L.iofs + rowbase + ixc;
        int valsum = (int)(__ldg(wb + c00) - __ldg(wb + c10) - __ldg(wb + c01) + __ldg(wb + c11));
        uint32_t valsq = __ldg(qb + c00) - __ldg(qb + c10) - __ldg(qb + c01) + __ldg(qb + c11);
        double nf = __dsub_rn(__dmul_rn(area, (double)valsq), __dmul_rn((double)valsum, (double)valsum));
        float vnf = 0.f;
        bool ok = false;
        if (nf > 0.) {
            vnf = __double2float_rn(__ddiv_rn(1.0, __dsqrt_rn(nf)));
            ok = __dmul_rn(area, (double)vnf) < 1e-1;
        }
        bool fail = false;
        if (ok) {
            double tmp = 0.;
            for (int i = 0; i < n0; i++) {
                StumpRegs s = load_stump(stumps + i);
                tmp = __dadd_rn(tmp, (double)stump_leaf(wb, v, s, vnf));
            }
            fail = tmp < thr0;
        }
        ok = ok && valid;
        fail = fail && ok;
        uint32_t f = __ballot_sync(0xffffffffu, fail);
        // e[i+1] = !(e[i] && stage0_failed[i]); every lane runs the same 32-step automaton
        uint32_t em = 0;
#pragma unroll
        for (int i = 0; i < 32; i++) {
            em |= (uint32_t)e << i;
            e = !(e && ((f >> i) & 1u));
        }
        bool visited = (em >> lane) & 1u;
        bool alive = visited && ok && !fail;
        uint32_t am = __ballot_sync(0xffffffffu, alive);
        nalive += __popc(am);
        if (lane == 0) bits_alive[L.bofs + iy * L.nxw + cx] = am;
        if (alive) vnf_out[L.wofs + iy * L.nx + ix] = vnf;
        if (depth && valid && !alive)
            depth[L.wofs + iy * L.nx + ix] = (int16_t)(!visited ? NV_DEPTH_SKIPPED : (!ok ? NV_DEPTH_VARREJ : 0));
    }
    if (lane == 0 && nalive) atomicAdd(&counters[0], nalive);
}

// Same pass with every level-dependent offset precomputed on the host and passed in the parameter bank: the
// address arithmetic is warp-uniform (uniform datapath), and the 32-step automaton is replaced by its closed
// form on bit-words.  Let g[i] = "window i was visited and failed stage 0"; then g[i+1] = f[i+1] & !g[i], i.e. inside
// every run of consecutive failures g is set at even offsets from the run start (a carry-in skip just removes
// bit 0 from the first run); visited[i+1] = !g[i].  Runs starting at even / odd positions are isolated with one
// addition each (the carry clears exactly the run it enters).
__device__ __forceinline__ uint32_t skip_rule_word(uint32_t f, bool &e)
{
    uint32_t fp = e ? f : (f & ~1u);
    uint32_t s = fp & ~(fp << 1);
    uint32_t me = fp & ~(fp + (s & 0x55555555u)), mo = fp & ~(fp + (s & 0xAAAAAAAAu));
    uint32_t g = (me & 0x55555555u) | (mo & 0xAAAAAAAAu);
    uint32_t em = (~(g << 1) & ~1u) | (e ? 1u : 0u);
    e = !(g >> 31);
    return em;
}

// BATCH: image blockIdx.y; integrals, vnf and alive bits at its strides, its alive count in its own counter block
// (P.counters + 16 * (1 + image)); queue entries are (image << 14) | dense window index, the queue and its count shared.
template <bool BATCH>
__global__ void __launch_bounds__(256) k_stage0_rows_p(const __grid_constant__ Stage0Params P)
{
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * 8 + uniformize_s0(threadIdx.x >> 5);
    if (row >= P.total_rows) return;
    const uint32_t *sum = P.sum, *sq = P.sq;
    float *vnfs = P.vnf;
    uint32_t *bits_alive = P.bits_alive;
    int *cnt = P.counters;
    if (BATCH) {
        sum += blockIdx.y * P.integ_stride; sq += blockIdx.y * P.integ_stride;
        vnfs += blockIdx.y * (size_t)P.win_stride; bits_alive += blockIdx.y * (size_t)P.bits_stride;
        cnt += 16 * (1 + blockIdx.y);
    }
    int l = 0;
    while (l + 1 < P.nlevels && P.lv_a[l + 1].x <= row) l++;
    const int4 la = P.lv_a[l], lb = P.lv_b[l], vr = P.var[l];
    const int iy = row - la.x, nxw = la.y, nx = la.z;
    const uint32_t *srow = sum + lb.x + (size_t)iy * la.w, *qrow = sq + lb.x + (size_t)iy * la.w;
    const double area = (double)((P.win_w - 2) * (P.win_h - 2));
    const double thr0 = (double)P.thr0;
    bool e = true;                                   // is the next window visited?  (x = 0 always is)
    int nalive = 0;
    for (int cx = 0; cx < nxw; cx++) {
        int ix = cx * 32 + lane;
        bool valid = ix < nx;
        int ixc = valid ? ix : nx - 1;
        const uint32_t *wb = srow + ixc, *qb = qrow + ixc;
        int valsum = (int)(__ldg(wb + vr.x) - __ldg(wb + vr.y) - __ldg(wb + vr.z) + __ldg(wb + vr.w));
        uint32_t valsq = __ldg(qb + vr.x) - __ldg(qb + vr.y) - __ldg(qb + vr.z) + __ldg(qb + vr.w);
        double nf = __dsub_rn(__dmul_rn(area, (double)valsq), __dmul_rn((double)valsum, (double)valsum));
        float vnf = 0.f;
        bool ok = false;
        if (nf > 0.) {
            vnf = __double2float_rn(__ddiv_rn(1.0, __dsqrt_rn(nf)));
            ok = __dmul_rn(area, (double)vnf) < 1e-1;
        }
        double tmp = 0.;
        for (int k = 0; k < P.n0; k++) {
            uint4 o0 = P.off[l][k][0], o1 = P.off[l][k][1];
            float2 w01 = P.cf[k][0], w2t = P.cf[k][1], lr = P.cf[k][2];
            int r0 = (int)(__ldg(wb + o0.x) - __ldg(wb + o0.y) - __ldg(wb + o0.z) + __ldg(wb + o0.w));
            int r1 = (int)(__ldg(wb + o1.x) - __ldg(wb + o1.y) - __ldg(wb + o1.z) + __ldg(wb + o1.w));
            float f = __fadd_rn(__fmul_rn(w01.x, __int2float_rn(r0)), __fmul_rn(w01.y, __int2float_rn(r1)));
            if (w2t.x != 0.f) {
                uint4 o2 = P.off[l][k][2];
                int r2 = (int)(__ldg(wb + o2.x) - __ldg(wb + o2.y) - __ldg(wb + o2.z) + __ldg(wb + o2.w));
                f = __fadd_rn(f, __fmul_rn(w2t.x, __int2float_rn(r2)));
            }
            f = __fmul_rn(f, vnf);
            tmp = __dadd_rn(tmp, (double)(f < w2t.y ? lr.x : lr.y));
        }
        ok = ok && valid;
        bool fail = ok && tmp < thr0;
        uint32_t fm = __ballot_sync(0xffffffffu, fail);
        uint32_t em = skip_rule_word(fm, e);
        bool visited = (em >> lane) & 1u;
        bool alive = visited && ok && !fail;
        uint32_t am = __ballot_sync(0xffffffffu, alive);
        nalive += __popc(am);
        if (lane == 0) bits_alive[lb.z + iy * nxw + cx] = am;
        if (alive) vnfs[lb.y + iy * nx + ix] = vnf;
        if (P.queue && am) {                             // small plan: k_alive_to_queue's job, without its launch
            int base = 0;
            if (lane == 0) base = atomicAdd(&P.counters[P.queue_cidx], __popc(am));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (alive) {
                const int pos = base + __popc(am & ((1u << lane) - 1u));
                const uint32_t id = BATCH ? ((uint32_t)blockIdx.y << 14) | (uint32_t)(lb.y + iy * nx + ix)
                                          : ((uint32_t)l << 26) | ((uint32_t)iy << 13) | (uint32_t)ix;
                if (pos < P.queue_cap) P.queue[pos] = make_uint2(id, __float_as_uint(vnf));
                else P.counters[2] = 1;
            }
        }
        if (P.depth && valid && !alive)
            P.depth[lb.y + iy * nx + ix] = (int16_t)(!visited ? NV_DEPTH_SKIPPED : (!ok ? NV_DEPTH_VARREJ : 0));
    }
    if (lane == 0 && nalive) atomicAdd(&cnt[0], nalive);
}

bool fill_stage0_params(const nv_cascade *c, const PlanDev &P, Stage0Params *sp)
{
    const DevCascade &m = c->meta;
    int n0 = m.stage_first[1];
    if (n0 > NV_S0_MAX_STUMPS || P.nlevels > NV_MAX_LEVELS) return false;
    sp->nlevels = P.nlevels; sp->total_rows = P.total_rows; sp->n0 = n0; sp->win_w = m.win_w; sp->win_h = m.win_h;
    sp->thr0 = m.stage_thr[0];
    for (int k = 0; k < n0; k++) {
        const DevStump &d = c->stumps[k];
        sp->cf[k][0] = make_float2(d.w[0], d.w[1]);
        sp->cf[k][1] = make_float2(d.w[2], d.thr);
        sp->cf[k][2] = make_float2(d.left, d.right);
    }
    for (int l = 0; l < P.nlevels; l++) {
        const LevelDesc &L = P.lv[l];
        auto off = [&](int dx, int dy) { return (uint32_t)(dy * L.ipitch + (L.ystep == 2 ? (dx & 1) * L.iplane + (dx >> 1) : dx)); };
        for (int k = 0; k < n0; k++)
            for (int j = 0; j < 3; j++) {
                uint32_t r = c->stumps[k].r[j];
                int x = r & 255, y = (r >> 8) & 255, w = (r >> 16) & 255, h = r >> 24;
                sp->off[l][k][j] = make_uint4(off(x, y), off(x + w, y), off(x, y + h), off(x + w, y + h));
            }
        sp->var[l] = make_int4((int)off(1, 1), (int)off(m.win_w - 1, 1), (int)off(1, m.win_h - 1), (int)off(m.win_w - 1, m.win_h - 1));
        sp->lv_a[l] = make_int4(L.row0, L.nxw, L.nx, L.ystep * L.ipitch);
        sp->lv_b[l] = make_int4(L.iofs, L.wofs, L.bofs, 0);
    }
    return true;
}

// expands alive bit-words into a window queue (fallback path for cascades the tile kernel cannot take)
__global__ void __launch_bounds__(256)
k_alive_to_queue(const PlanDev *__restrict__ plan, int total_rows, const float *__restrict__ vnf,
                 const uint32_t *__restrict__ bits_alive, uint2 *__restrict__ queue, int *__restrict__ counters,
                 int queue_cap, int cidx)
{
    int lane = threadIdx.x & 31;
    int row = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= total_rows) return;
    int l = find_level_c(plan, row, &LevelDesc::row0);
    const LevelDesc &L = plan->lv[l];
    int iy = row - L.row0;
    for (int cx = 0; cx < L.nxw; cx++) {
        uint32_t am = bits_alive[L.bofs + iy * L.nxw + cx];
        if (!am) continue;
        int base = 0;
        if (lane == 0) base = atomicAdd(&counters[cidx], __popc(am));
        base = __shfl_sync(0xffffffffu, base, 0);
        if ((am >> lane) & 1u) {
            int ix = cx * 32 + lane, pos = base + __popc(am & ((1u << lane) - 1u));
            if (pos < queue_cap)
                queue[pos] = make_uint2(((uint32_t)l << 26) | ((uint32_t)iy << 13) | (uint32_t)ix,
                                        __float_as_uint(vnf[L.wofs + iy * L.nx + ix]));
            else
                counters[2] = 1;
        }
    }
}

// ---- TMA / mbarrier primitives (sm_90+ PTX; SASS: UTMALDG, SYNCS) ------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t phase)
{
    uint32_t done;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(bar), "r"(phase) : "memory");
    } while (!done);
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *map, int x, int y, uint32_t bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(x), "r"(y) : "memory");
}

// A value that is the same in every lane, rebuilt from warp votes so that the compiler can PROVE it is
// warp-uniform (vote results are) and keep loop control on the uniform datapath.
__device__ __forceinline__ int uniformize(int v, int bits)
{
    int r = 0;
    for (int k = 0; k < bits; k++) r |= (int)(__ballot_sync(0xffffffffu, (v >> k) & 1) & (1u << k));
    return r;
}

// ================================================================================================
// k_cascade_classes — the bulk stages, free of shared-memory bank conflicts.
// A tile is NV_CTX x NV_CTY = 64 x 32 windows; its integral patch (+halo) is staged in shared memory by TMA, one
// 2-D box per column plane.  The tile's pitch makes the bank of every corner read of window (lx, ly) equal to
// (lx + kskew * ly + const) mod 32, so the 2048 windows fall into 32 bank classes of 64 members (member index =
// 2 * ly + lx / 32).  Lane c of every warp only ever evaluates windows of class c: the 32 lanes of a corner load hit
// 32 different banks whatever the alive pattern is (the compacted-queue kernel this replaces spent 59 % of its
// shared-memory wavefronts on conflict replays, profiles/r1_v2_summary.md).  The alive set of a class is a 64-bit
// mask; in every stage warp w takes the set bits of rank w, w + 8, ..., so no queue and no compaction is needed, and
// the surviving bits are OR-ed into the next stage's mask.  The price is imbalance between classes (a round runs as
// long as the fullest class has members left): on config 3, 6.8 M warp rounds per frame against 5.1 M for perfect
// compaction, but each weak classifier costs 8.7 wavefronts instead of 22.
//
// FAST variant (certificates computed by fill_bulk_stumps): the cascade's stage sums are order-free and its feature
// weights are small integers.  Then (a) w0*r0 + w1*r1 (+ w2*r2) is evaluated in int32 and converted once — every
// float operation of the reference is exact on such values, so the result is the same float; (b) the stage sum starts
// at the sum of all right leaves and a classifier whose feature is below its threshold adds (left - right), one
// predicated DADD; (c) two-rect classifiers run before three-rect ones, each in a branch-free loop.  The general
// variant keeps the reference's float operations and XML order.
// ================================================================================================
#ifndef NV_CLS_UNROLL
#define NV_CLS_UNROLL 2            // weak classifiers in flight per lane in the bulk kernel's inner loops
#endif
constexpr int CLS_UNROLL = NV_CLS_UNROLL;

__device__ __forceinline__ uint32_t lds_u32(uint32_t addr)
{
    uint32_t v;
    asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ int rect4(uint32_t wa, const uint4 &o)
{
    return (int)(lds_u32(wa + o.x) - lds_u32(wa + o.y) - lds_u32(wa + o.z) + lds_u32(wa + o.w));
}
// minus the rect sum: b + c - a - d
__device__ __forceinline__ int nrect4(uint32_t wa, const uint4 &o)
{
    return (int)(lds_u32(wa + o.y) + lds_u32(wa + o.z) - lds_u32(wa + o.x) - lds_u32(wa + o.w));
}
// tmp += d if f < thr, in two instructions: FSET.BF yields the bits of 1.0f or 0, which as the HIGH word of a double
// (low word 0) read 2^-7 or 0.0; d128 = 128 * d, so the fused multiply-add adds exactly d or exactly 0.
__device__ __forceinline__ void add_if_lt(double &tmp, float f, float thr, double d128)
{
    float m = f < thr ? 1.0f : 0.0f;
    tmp = __fma_rn(d128, __hiloint2double(__float_as_int(m), 0), tmp);
}

// NW windows (1 or 2) of one lane through one stage; pass[i] = "stage passed"
template <bool FAST, int NW, typename PT>
__device__ __forceinline__ void class_stage(const PT &P, int si, const uint32_t (&wa)[NW], const float (&vnf)[NW],
                                            bool (&pass)[NW])
{
    const int k0 = P.stage_first[si], k1 = P.stage_first[si + 1];
    const double thr = (double)P.stage_thr[si];
    double tmp[NW];
    if (FAST) {
        const int k6 = P.stage_mid6[si], km = P.stage_mid[si];
#pragma unroll
        for (int i = 0; i < NW; i++) tmp[i] = P.stage_base[si];
#pragma unroll CLS_UNROLL
        for (int k = k0; k < k6; k++) {                         // two rects sharing two corners: six loads (fill_bulk_stumps)
            const BulkStump &S = P.s[k];
            const double d = __hiloint2double((int)S.d_hi, (int)S.d_lo);
            const float sthr = __uint_as_float(S.thr);
#pragma unroll
            for (int i = 0; i < NW; i++) {
                int u = (int)(lds_u32(wa[i] + S.o0.x) - lds_u32(wa[i] + S.o0.y));
                int nr0 = (int)(lds_u32(wa[i] + S.o0.z) - lds_u32(wa[i] + S.o0.w)) - u;
                int r1 = u - (int)lds_u32(wa[i] + S.o1.x) + (int)lds_u32(wa[i] + S.o1.y);
                add_if_lt(tmp[i], __fmul_rn(__int2float_rn((int)S.w1 * r1 + nr0), vnf[i]), sthr, d);
            }
        }
#pragma unroll CLS_UNROLL
        for (int k = k6; k < km; k++) {                         // two rects, eight loads
            const BulkStump &S = P.s[k];
            const double d = __hiloint2double((int)S.d_hi, (int)S.d_lo);
            const float sthr = __uint_as_float(S.thr);
#pragma unroll
            for (int i = 0; i < NW; i++) {
                int r = (int)S.w1 * rect4(wa[i], S.o1) + nrect4(wa[i], S.o0);
                add_if_lt(tmp[i], __fmul_rn(__int2float_rn(r), vnf[i]), sthr, d);
            }
        }
#pragma unroll CLS_UNROLL
        for (int k = km; k < k1; k++) {                         // three rects
            const BulkStump &S = P.s[k];
            const double d = __hiloint2double((int)S.d_hi, (int)S.d_lo);
            const float sthr = __uint_as_float(S.thr);
#pragma unroll
            for (int i = 0; i < NW; i++) {
                int r = (int)S.w1 * rect4(wa[i], S.o1) + (int)S.w2 * rect4(wa[i], P.o2[k]) + nrect4(wa[i], S.o0);
                add_if_lt(tmp[i], __fmul_rn(__int2float_rn(r), vnf[i]), sthr, d);
            }
        }
    } else {
#pragma unroll
        for (int i = 0; i < NW; i++) tmp[i] = 0.;
        for (int k = k0; k < k1; k++) {                         // XML order, the reference's float operations
            const BulkStump &S = P.s[k];
            const float w0 = __uint_as_float(S.w0), w1 = __uint_as_float(S.w1), w2 = __uint_as_float(S.w2);
            const float sthr = __uint_as_float(S.thr), left = __uint_as_float(S.left), right = __uint_as_float(S.right);
#pragma unroll
            for (int i = 0; i < NW; i++) {
                float f = __fadd_rn(__fmul_rn(w0, __int2float_rn(rect4(wa[i], S.o0))),
                                    __fmul_rn(w1, __int2float_rn(rect4(wa[i], S.o1))));
                if (w2 != 0.f) f = __fadd_rn(f, __fmul_rn(w2, __int2float_rn(rect4(wa[i], P.o2[k]))));
                f = __fmul_rn(f, vnf[i]);
                tmp[i] = __dadd_rn(tmp[i], (double)(f < sthr ? left : right));
            }
        }
    }
#pragma unroll
    for (int i = 0; i < NW; i++) pass[i] = !(tmp[i] < thr);
}

template <int YS, bool FAST>
__global__ void __launch_bounds__(256) k_cascade_classes(const __grid_constant__ TileParams P)
{
    extern __shared__ __align__(128) uint32_t tile[];           // [YS planes][rt][cp], plane stride ps
    __shared__ __align__(8) unsigned long long mbar;
    __shared__ uint32_t s_mask[3][2][32];                        // rotating alive masks: [buffer][member / 32][class]
    __shared__ uint32_t s_words[NV_CTY][2];
    const PlanDev *__restrict__ plan = P.plan;
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = uniformize(tid >> 5, 3);

    int t = blockIdx.x, l = P.level_begin;
    while (l + 1 < P.level_end && plan->lv[l + 1].ctile0 <= t) l++;
    const LevelDesc &L = plan->lv[l];
    int rel = t - L.ctile0, ty = rel / L.cntx, tx = rel - ty * L.cntx;
    int iy0 = ty * NV_CTY, ix0 = tx * NV_CTX;
    const int CP = P.cp, PS = P.ps, K = P.kskew;
    uint32_t bar = smem_u32(&mbar);

    if (tid == 0) mbar_init(bar, 1);
    if (tid < 64) {                                              // the tile's alive words, two per window row
        int ly = tid >> 1, cx = 2 * tx + (tid & 1);
        s_words[ly][tid & 1] = (iy0 + ly < L.ny && cx < L.nxw) ? P.bits_alive[L.bofs + (size_t)(iy0 + ly) * L.nxw + cx] : 0u;
    } else {
        (&s_mask[0][0][0])[tid - 64] = 0u;
    }
    __syncthreads();
    if (tid == 0) {                                              // stage the integral tile: one box per plane
        mbar_expect_tx(bar, (uint32_t)(YS * P.rt * CP * 4));
#pragma unroll
        for (int p = 0; p < YS; p++)
            tma_load_2d(smem_u32(tile + p * PS), P.maps + l, ix0 + p * L.iplane, iy0 * YS, bar);
    }
    {   // class masks: warp w transposes window rows 4w .. 4w+3 (8 members, all in the same mask half)
        uint32_t part = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            int ly = warp * 4 + (i >> 1), h = i & 1;
            uint32_t b = (s_words[ly][h] >> ((lane - K * ly) & 31)) & 1u;
            part |= b << ((ly * 2 + h) & 31);
        }
        if (part) atomicOr(&s_mask[0][warp >> 2][lane], part);
    }
    __syncthreads();
    mbar_wait(bar, 0);                                           // also before an early exit: the copy targets this CTA's smem

    const uint32_t tile_sa = smem_u32(tile);
    const float *__restrict__ vnf_tile = P.vnf + L.wofs + (size_t)iy0 * L.nx + ix0;
    const int rowb = YS * CP * 4;                                // bytes from one window row to the next
    int cur = 0;
    for (int st = P.stage_begin; st < P.stage_end; st++) {
        const int si = st - P.stage_begin;
        uint32_t mlo = s_mask[cur][0][lane], mhi = s_mask[cur][1][lane];
        int maxc = uniformize(__reduce_max_sync(0xffffffffu, __popc(mlo) + __popc(mhi)), 7);
        if (maxc == 0) return;                                   // block-uniform: every warp reads the same masks
        int nxt = cur == 2 ? 0 : cur + 1, zer = nxt == 2 ? 0 : nxt + 1;
        if (warp == 0) { s_mask[zer][0][lane] = 0u; s_mask[zer][1][lane] = 0u; }
        unsigned long long rem = ((unsigned long long)mhi << 32) | mlo, pass_bits = 0ull;
        for (int i = 0; i < warp; i++) rem &= rem - 1ull;        // warp w takes the set bits of rank w, w + 8, ...
        int j = warp;
        for (; j + 8 < maxc; j += 16) {                          // two windows per lane and round
            int bit[2]; bool active[2], pass[2]; uint32_t wa[2]; float vnf[2]; int ly[2], lx[2];
#pragma unroll
            for (int i = 0; i < 2; i++) {
                active[i] = rem != 0ull;
                bit[i] = active[i] ? __ffsll((long long)rem) - 1 : 0;
                ly[i] = bit[i] >> 1; lx[i] = ((lane - K * ly[i]) & 31) + ((bit[i] & 1) << 5);
                wa[i] = tile_sa + (uint32_t)(ly[i] * rowb + lx[i] * 4);
                vnf[i] = active[i] ? __ldg(vnf_tile + ly[i] * L.nx + lx[i]) : 0.f;     // per-window factor, L2-resident
#pragma unroll
                for (int q = 0; q < 8; q++) rem &= rem - 1ull;
            }
            class_stage<FAST, 2>(P, si, wa, vnf, pass);
#pragma unroll
            for (int i = 0; i < 2; i++) {
                if (active[i] && pass[i]) pass_bits |= 1ull << bit[i];
                if (P.depth && active[i] && !pass[i]) P.depth[L.wofs + (iy0 + ly[i]) * L.nx + ix0 + lx[i]] = (int16_t)(-st);
            }
        }
        for (; j < maxc; j += 8) {                               // at most one single-window round
            bool active = rem != 0ull;
            int bit = active ? __ffsll((long long)rem) - 1 : 0;
            int ly = bit >> 1, lx = ((lane - K * ly) & 31) + ((bit & 1) << 5);
            uint32_t wa[1] = {tile_sa + (uint32_t)(ly * rowb + lx * 4)};
            float vnf[1] = {active ? __ldg(vnf_tile + ly * L.nx + lx) : 0.f};
            bool pass[1];
            class_stage<FAST, 1>(P, si, wa, vnf, pass);
            if (active && pass[0]) pass_bits |= 1ull << bit;
            if (P.depth && active && !pass[0]) P.depth[L.wofs + (iy0 + ly) * L.nx + ix0 + lx] = (int16_t)(-st);
#pragma unroll
            for (int q = 0; q < 8; q++) rem &= rem - 1ull;
        }
        if ((uint32_t)pass_bits) atomicOr(&s_mask[nxt][0][lane], (uint32_t)pass_bits);
        if ((uint32_t)(pass_bits >> 32)) atomicOr(&s_mask[nxt][1][lane], (uint32_t)(pass_bits >> 32));
        __syncthreads();
        cur = nxt;
    }
    // survivors: candidates if the bulk stages were the whole cascade, else the tail queue
    if (warp != 0) return;
    uint32_t mlo = s_mask[cur][0][lane], mhi = s_mask[cur][1][lane];
    int cnt = __popc(mlo) + __popc(mhi), inc = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        int v = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += v;
    }
    int total = __shfl_sync(0xffffffffu, inc, 31);
    if (total == 0) return;
    int *counter = P.counters + (P.final_stage ? 1 : 3);
    int cap = P.final_stage ? P.cand_cap : P.tail_cap;
    int base = 0;
    if (lane == 0) base = atomicAdd(counter, total);
    base = __shfl_sync(0xffffffffu, base, 0) + inc - cnt;
    unsigned long long rem = ((unsigned long long)mhi << 32) | mlo;
    for (; rem; rem &= rem - 1ull, base++) {
        int bit = __ffsll((long long)rem) - 1;
        int ly = bit >> 1, lx = ((lane - K * ly) & 31) + ((bit & 1) << 5);
        uint32_t key = ((uint32_t)l << 26) | ((uint32_t)(iy0 + ly) << 13) | (uint32_t)(ix0 + lx);
        if (base >= cap) { P.counters[2] = 1; continue; }
        if (P.final_stage) {
            P.cand[base] = key;
            if (P.depth) P.depth[L.wofs + (iy0 + ly) * L.nx + ix0 + lx] = NV_DEPTH_PASS;
        } else
            P.tail[base] = make_uint2(key, __float_as_uint(__ldg(vnf_tile + ly * L.nx + lx)));
    }
}

// ================================================================================================
// k_cascade_wide — the bulk stages on WIDE tiles (round 2; ystep-1 levels).  Same bank-class scheme as k_cascade_classes
// — lane c only evaluates windows of class (lx + kskew * ly) & 31, so corner loads never conflict — but the tile is
// TW x TH windows with TW * TH / 32 = 128 or 256 members per class.  A stage costs "members of the fullest class" warp
// steps per weak classifier, so the more members a class has the closer the fullest class is to the average one: on
// config 3 the ystep-1 levels take 4.30 M steps in 64x32 tiles, 3.83 M in 64x64 and 3.49 M in 128x64 (simulated on the
// oracle's depth maps; the 64x32 figure equals the DFMA count ncu reports for k_cascade_classes<1>).
// What changes with the mask width is how a warp finds its windows.  The alive set of a class is TW * TH / 1024 words in
// shared memory; warp w takes the CONTIGUOUS ranks [w q, (w + 1) q), q = ceil(fullest class / warps) — the same steps per
// warp as the interleaved ranks of k_cascade_classes, but a lane walks its words once: skip w q set bits at the start of
// the stage, then one "clear lowest bit" per window instead of eight.
// ================================================================================================
template <int YS, bool FAST, int TW, int TH, int NWARP>
__global__ void __launch_bounds__(32 * NWARP) k_cascade_wide(const __grid_constant__ TileParams P)
{
    constexpr int HW = TW / 32;                                  // 32-window words per tile row
    constexpr int NM = TH * HW;                                  // members per class
    constexpr int MW = NM / 32;                                  // mask words per class
    constexpr int MPW = NM / NWARP;                              // members whose rows one warp transposes
    constexpr int NT = 32 * NWARP;
    static_assert(MPW <= 32 && 32 % MPW == 0 && TH % NWARP == 0 && (NWARP == 8 || NWARP == 16), "a warp's rows fill (part of) one mask word");
    extern __shared__ __align__(128) uint32_t tile[];           // [YS planes][rt][cp], plane stride ps
    __shared__ __align__(8) unsigned long long mbar;
    __shared__ uint32_t s_mask[3][MW][32];                       // rotating alive masks: [buffer][word][class]
    __shared__ uint32_t s_words[TH][HW];
    const PlanDev *__restrict__ plan = P.plan;
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = uniformize(tid >> 5, NWARP == 16 ? 4 : 3);

    int t = blockIdx.x, l = P.level_begin;
    while (l + 1 < P.level_end && plan->lv[l + 1].wtile0 <= t) l++;
    const LevelDesc &L = plan->lv[l];
    const int rel = t - L.wtile0, ty = rel / L.wntx, tx = rel - ty * L.wntx;
    const int iy0 = ty * TH, ix0 = tx * TW;
    const int CP = P.cp, PS = P.ps, K = P.kskew;
    const uint32_t bar = smem_u32(&mbar);

    if (tid == 0) mbar_init(bar, 1);
    for (int i = tid; i < TH * HW; i += NT) {                   // the tile's alive words
        const int ly = i / HW, h = i - ly * HW, cx = HW * tx + h;
        s_words[ly][h] = (iy0 + ly < L.ny && cx < L.nxw) ? P.bits_alive[L.bofs + (size_t)(iy0 + ly) * L.nxw + cx] : 0u;
    }
    for (int i = tid; i < 3 * MW * 32; i += NT) (&s_mask[0][0][0])[i] = 0u;
    __syncthreads();
    if (tid == 0) {                                              // stage the integral tile: one box per plane
        mbar_expect_tx(bar, (uint32_t)(YS * P.rt * CP * 4));
#pragma unroll
        for (int p = 0; p < YS; p++)
            tma_load_2d(smem_u32(tile + p * PS), P.maps + l, ix0 + p * L.iplane, iy0 * YS, bar);
    }
    {   // class masks: warp w transposes window rows [w TH / NWARP, (w + 1) TH / NWARP): MPW consecutive members of every class
        uint32_t part = 0;
#pragma unroll
        for (int i = 0; i < MPW; i++) {
            const int ly = warp * (TH / NWARP) + i / HW, h = i % HW;
            const uint32_t b = (s_words[ly][h] >> ((lane - K * ly) & 31)) & 1u;
            part |= b << i;
        }
        const int m0 = warp * MPW;
        if (part) atomicOr(&s_mask[0][m0 >> 5][lane], part << (m0 & 31));
    }
    __syncthreads();
    mbar_wait(bar, 0);                                           // also before an early exit: the copy targets this CTA's smem

    const uint32_t tile_sa = smem_u32(tile);
    const float *__restrict__ vnf_tile = P.vnf + L.wofs + (size_t)iy0 * L.nx + ix0;
    const int rowb = YS * CP * 4;                                // bytes from one window row to the next
    int cur = 0;
    for (int st = P.stage_begin; st < P.stage_end; st++) {
        const int si = st - P.stage_begin;
        int cnt = 0;
#pragma unroll
        for (int w = 0; w < MW; w++) cnt += __popc(s_mask[cur][w][lane]);
        const int maxc = uniformize(__reduce_max_sync(0xffffffffu, cnt), 9);
        if (maxc == 0) return;                                   // block-uniform: every warp reads the same masks
        const int nxt = cur == 2 ? 0 : cur + 1, zer = nxt == 2 ? 0 : nxt + 1;
        if (warp == 0) {
#pragma unroll
            for (int w = 0; w < MW; w++) s_mask[zer][w][lane] = 0u;
        }
        const int q = (maxc + NWARP - 1) / NWARP;                // ranks per warp: warp w takes [w q, (w + 1) q)
        int skip = warp * q;
        int mine = min(max(cnt - skip, 0), q);                   // windows of this lane in this stage
        const int steps = uniformize(min(max(maxc - skip, 0), q), 6);   // = the largest `mine` of the warp
        int wi = 0;
        uint32_t curw = 0u;
        if (mine > 0) {                                          // walk to the first of them
            curw = s_mask[cur][0][lane];
            for (int pc = __popc(curw); skip >= pc; pc = __popc(curw)) { skip -= pc; curw = s_mask[cur][++wi][lane]; }
            for (; skip > 0; skip--) curw &= curw - 1u;
        }
        for (int r = 0; r < steps; r += 2) {                     // two windows per lane and round
            int m[2], ly[2], lx[2]; bool active[2], pass[2]; uint32_t wa[2]; float vnf[2];
#pragma unroll
            for (int i = 0; i < 2; i++) {
                active[i] = mine > 0;
                m[i] = 0;
                if (active[i]) {
                    while (curw == 0u) curw = s_mask[cur][++wi][lane];
                    m[i] = (wi << 5) + __ffs((int)curw) - 1;
                    curw &= curw - 1u;
                    mine--;
                }
                ly[i] = m[i] / HW; lx[i] = ((lane - K * ly[i]) & 31) + ((m[i] % HW) << 5);
                wa[i] = tile_sa + (uint32_t)(ly[i] * rowb + lx[i] * 4);
                vnf[i] = active[i] ? __ldg(vnf_tile + ly[i] * L.nx + lx[i]) : 0.f;     // per-window factor, L2-resident
            }
            if (r + 1 < steps) class_stage<FAST, 2>(P, si, wa, vnf, pass);
            else {
                const uint32_t wa1[1] = {wa[0]}; const float vnf1[1] = {vnf[0]}; bool pass1[1];
                class_stage<FAST, 1>(P, si, wa1, vnf1, pass1);
                pass[0] = pass1[0]; pass[1] = false;
            }
#pragma unroll
            for (int i = 0; i < 2; i++) {
                if (active[i] && pass[i]) atomicOr(&s_mask[nxt][m[i] >> 5][lane], 1u << (m[i] & 31));
                if (P.depth && active[i] && !pass[i]) P.depth[L.wofs + (iy0 + ly[i]) * L.nx + ix0 + lx[i]] = (int16_t)(-st);
            }
        }
        __syncthreads();
        cur = nxt;
    }
    // survivors: candidates if the bulk stages were the whole cascade, else the tail queue
    if (warp != 0) return;
    int cnt = 0;
#pragma unroll
    for (int w = 0; w < MW; w++) cnt += __popc(s_mask[cur][w][lane]);
    int inc = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        int v = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += v;
    }
    const int total = __shfl_sync(0xffffffffu, inc, 31);
    if (total == 0) return;
    int *counter = P.counters + (P.final_stage ? 1 : 3);
    const int cap = P.final_stage ? P.cand_cap : P.tail_cap;
    int base = 0;
    if (lane == 0) base = atomicAdd(counter, total);
    base = __shfl_sync(0xffffffffu, base, 0) + inc - cnt;
    for (int w = 0; w < MW; w++) {
        for (uint32_t rem = s_mask[cur][w][lane]; rem; rem &= rem - 1u, base++) {
            const int m = (w << 5) + __ffs((int)rem) - 1;
            const int ly = m / HW, lx = ((lane - K * ly) & 31) + ((m % HW) << 5);
            const uint32_t key = ((uint32_t)l << 26) | ((uint32_t)(iy0 + ly) << 13) | (uint32_t)(ix0 + lx);
            if (base >= cap) { P.counters[2] = 1; continue; }
            if (P.final_stage) {
                P.cand[base] = key;
                if (P.depth) P.depth[L.wofs + (iy0 + ly) * L.nx + ix0 + lx] = NV_DEPTH_PASS;
            } else
                P.tail[base] = make_uint2(key, __float_as_uint(__ldg(vnf_tile + ly * L.nx + lx)));
        }
    }
}

// ================================================================================================
// k_stage0_tiles + k_stage0_chain — variance normalisation and stage 0 of a LARGE plan (FAST cascades), round 2.
// k_stage0_rows_p reads its ~44 integral words per window from global memory with a 64-bit address formed for each
// (343 warp instructions per 32 windows: 46 M per config-3 frame, 14 % of the frame's issue work).  Here stage 0 runs on
// the bulk kernel's tiles instead: the integral tile comes in by TMA, every lane is bound to its bank class, all 64
// members of every class are evaluated (nothing is known about the windows yet, so the schedule is dense and the lane
// use perfect), two windows per lane share the uniform classifier loads, features in int32.  The skip rule needs the
// failures of a whole window row in order, so this kernel only writes two bits per window — "valid and passes the
// variance test" and "failed stage 0" — plus the factor; k_stage0_chain then runs the rule along every row on those
// bit-words (a warp per row, the 32-window words of a row in parallel: each word maps the incoming "next window is
// visited" flag to the outgoing one, and the prefix of that composition is a five-step shuffle scan).
// ================================================================================================
template <int YS>
__global__ void __launch_bounds__(256) k_stage0_tiles(const __grid_constant__ Stage0TileParams P)
{
    extern __shared__ __align__(128) uint32_t tile[];
    __shared__ __align__(8) unsigned long long mbar;
    const PlanDev *__restrict__ plan = P.plan;
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = uniformize(tid >> 5, 3);
    int t = blockIdx.x, l = P.level_begin;
    while (l + 1 < P.level_end && plan->lv[l + 1].ctile0 <= t) l++;
    const LevelDesc &L = plan->lv[l];
    const int rel = t - L.ctile0, ty = rel / L.cntx, tx = rel - ty * L.cntx;
    const int iy0 = ty * NV_CTY, ix0 = tx * NV_CTX;
    const int CP = P.cp, PS = P.ps, K = P.kskew;
    const uint32_t bar = smem_u32(&mbar);
    if (tid == 0) mbar_init(bar, 1);
    __syncthreads();
    if (tid == 0) {
        mbar_expect_tx(bar, (uint32_t)(YS * P.rt * CP * 4));
#pragma unroll
        for (int p = 0; p < YS; p++)
            tma_load_2d(smem_u32(tile + p * PS), P.maps + l, ix0 + p * L.iplane, iy0 * YS, bar);
    }
    // the squared integral is read from global memory: four corners per window, nothing else uses it
    const int ww = P.win_w, wh = P.win_h;
    auto gcorner = [&](int dx, int dy) { return dy * L.ipitch + (YS == 2 ? (dx & 1) * L.iplane + (dx >> 1) : dx); };
    const int q00 = gcorner(1, 1), q10 = gcorner(ww - 1, 1), q01 = gcorner(1, wh - 1), q11 = gcorner(ww - 1, wh - 1);
    const uint32_t *__restrict__ sqb = P.sq + L.iofs;
    const double area = (double)((ww - 2) * (wh - 2));
    const uint32_t tile_sa = smem_u32(tile);
    const int rowb = YS * CP * 4;
    mbar_wait(bar, 0);
#pragma unroll 1
    for (int r = 0; r < 4; r++) {                                // warp w: window rows 4w .. 4w + 3, both halves of a row per round
        const int ly = warp * 4 + r, iy = iy0 + ly;
        const int iyc = min(iy, L.ny - 1);
        uint32_t wa[2]; float vnf[2]; bool ok[2], pass[2]; int lx[2];
#pragma unroll
        for (int h = 0; h < 2; h++) {
            lx[h] = ((lane - K * ly) & 31) + (h << 5);
            wa[h] = tile_sa + (uint32_t)(ly * rowb + lx[h] * 4);
            const int ixc = min(ix0 + lx[h], L.nx - 1);
            const uint32_t *qb = sqb + (size_t)iyc * YS * L.ipitch + ixc;
            const int valsum = (int)(lds_u32(wa[h] + P.var.x) - lds_u32(wa[h] + P.var.y) - lds_u32(wa[h] + P.var.z) + lds_u32(wa[h] + P.var.w));
            const uint32_t valsq = __ldg(qb + q00) - __ldg(qb + q10) - __ldg(qb + q01) + __ldg(qb + q11);
            const double nf = __dsub_rn(__dmul_rn(area, (double)valsq), __dmul_rn((double)valsum, (double)valsum));
            vnf[h] = 0.f; ok[h] = false;
            if (nf > 0.) {
                vnf[h] = __double2float_rn(__ddiv_rn(1.0, __dsqrt_rn(nf)));
                ok[h] = __dmul_rn(area, (double)vnf[h]) < 1e-1;
            }
            ok[h] = ok[h] && iy < L.ny && ix0 + lx[h] < L.nx;
        }
        class_stage<true, 2>(P, 0, wa, vnf, pass);
        const int rot = (K * ly) & 31;                           // lane j holds the window at bit (j - K ly) & 31 of its word
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const uint32_t om = __ballot_sync(0xffffffffu, ok[h]), fm = __ballot_sync(0xffffffffu, ok[h] && !pass[h]);
            const int cx = 2 * tx + h;
            if (iy < L.ny && cx < L.nxw) {
                if (lane == 0) {
                    const size_t wi = (size_t)L.bofs + (size_t)iy * L.nxw + cx;
                    P.bits_okv[wi] = __funnelshift_r(om, om, rot);
                    P.bits_fail[wi] = __funnelshift_r(fm, fm, rot);
                }
                if (ok[h]) P.vnf[L.wofs + (size_t)iy * L.nx + ix0 + lx[h]] = vnf[h];
            }
        }
    }
}

// the level table of a plan as k_stage0_chain reads it: in the kernel's parameter (constant) bank, so that finding a
// row's level is a walk over uniform loads and not a chain of dependent global ones (18 us of latency for the last levels)
struct ChainParams {
    int4 a[NV_MAX_LEVELS];         // row0, nxw, nx, bofs
    int wofs[NV_MAX_LEVELS];
    int nlevels, total_rows;
    const uint32_t *bits_fail, *bits_okv;
    uint32_t *bits_alive;
    int *counters;
    int16_t *depth;
};

__global__ void __launch_bounds__(256) k_stage0_chain(const __grid_constant__ ChainParams P)
{
    const uint32_t *__restrict__ bits_fail = P.bits_fail, *__restrict__ bits_okv = P.bits_okv;
    uint32_t *__restrict__ bits_alive = P.bits_alive;
    int16_t *__restrict__ depth = P.depth;
    int *__restrict__ counters = P.counters;
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * 8 + uniformize_s0(threadIdx.x >> 5);
    if (row >= P.total_rows) return;
    int l = 0;
    while (l + 1 < P.nlevels && P.a[l + 1].x <= row) l++;
    struct { int row0, nxw, nx, bofs, wofs; } L = {P.a[l].x, P.a[l].y, P.a[l].z, P.a[l].w, P.wofs[l]};
    const int iy = row - L.row0;
    const size_t wbase = (size_t)L.bofs + (size_t)iy * L.nxw;
    bool carry = true;                                           // x = 0 is always visited
    int nalive = 0;
    for (int c0 = 0; c0 < L.nxw; c0 += 32) {
        const int cx = c0 + lane;
        const bool have = cx < L.nxw;
        const uint32_t f = have ? bits_fail[wbase + cx] : 0u, o = have ? bits_okv[wbase + cx] : 0u;
        bool e0 = false, e1 = true;
        const uint32_t em0 = skip_rule_word(f, e0), em1 = skip_rule_word(f, e1);   // e0 / e1: flag after this word for an incoming 0 / 1
        bool a = e0, b = e1;                                     // inclusive scan of the composition: (out for 0, out for 1) of words 0 .. lane
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const bool pa = __shfl_up_sync(0xffffffffu, (int)a, d), pb = __shfl_up_sync(0xffffffffu, (int)b, d);
            if (lane >= d) { const bool na = pa ? b : a, nb = pb ? b : a; a = na; b = nb; }
        }
        const bool xa = __shfl_up_sync(0xffffffffu, (int)a, 1), xb = __shfl_up_sync(0xffffffffu, (int)b, 1);
        const bool ein = lane == 0 ? carry : (carry ? xb : xa);
        const uint32_t em = ein ? em1 : em0;
        const uint32_t alive = em & o & ~f;
        if (have) bits_alive[wbase + cx] = alive;
        nalive += __popc(alive);
        if (depth && have) {
            for (int j = 0; j < 32; j++) {
                const int ix = cx * 32 + j;
                if (ix < L.nx && !((alive >> j) & 1u))
                    depth[L.wofs + (size_t)iy * L.nx + ix] = (int16_t)(!((em >> j) & 1u) ? NV_DEPTH_SKIPPED : (!((o >> j) & 1u) ? NV_DEPTH_VARREJ : 0));
            }
        }
        const bool la = __shfl_sync(0xffffffffu, (int)a, 31), lb = __shfl_sync(0xffffffffu, (int)b, 31);
        carry = carry ? lb : la;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) nalive += __shfl_xor_sync(0xffffffffu, nalive, d);
    if (lane == 0 && nalive) atomicAdd(&counters[0], nalive);
}

#define TAIL_MAX_WIN 32
__global__ void __launch_bounds__(256)
k_cascade_tail(const PlanDev *__restrict__ plan, const DevCascade *__restrict__ meta, const DevStump *__restrict__ stumps,
               const uint32_t *__restrict__ sum, const uint2 *__restrict__ tail, int *__restrict__ counters,
               uint32_t *__restrict__ cand, int cand_cap, int16_t *__restrict__ depth, int stage_begin, int order_free)
{
    extern __shared__ uint32_t s_win[];                          // 8 warps x (win_h+1) x (win_w+1) words
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int n = counters[3], nstages = meta->nstages;
    int ww = plan->win_w, wh = plan->win_h, LP = ww + 1, npatch = (wh + 1) * LP;
    uint32_t *win = s_win + warp * npatch;
    for (;;) {                                                   // windows are handed out one at a time: depths are very uneven
        int e = 0;
        if (lane == 0) e = atomicAdd(&counters[5], 1);
        e = __shfl_sync(0xffffffffu, e, 0);
        if (e >= n) break;
        uint2 q = tail[e];
        int l = q.x >> 26, iy = (q.x >> 13) & 8191, ix = q.x & 8191;
        float vnf = __uint_as_float(q.y);
        const LevelDesc &L = plan->lv[l];
        const uint32_t *wb = sum + L.iofs + (size_t)iy * L.ystep * L.ipitch + ix;
        __syncwarp();
        for (int idx = lane; idx < npatch; idx += 32) {          // private copy of the window's integral patch
            int r = idx / LP, c = idx - r * LP;
            int pc = L.ystep == 2 ? (c & 1) * L.iplane + (c >> 1) : c;
            win[idx] = __ldg(wb + (size_t)r * L.ipitch + pc);
        }
        __syncwarp();
        int code = NV_DEPTH_PASS;
        for (int st = stage_begin; st < nstages; st++) {
            int k0 = meta->stage_first[st], k1 = meta->stage_first[st + 1];
            double tmp = 0.;
            for (int kb = k0; kb < k1; kb += 32) {               // 32 weak classifiers per round, one per lane
                int k = kb + lane;
                double leaf = 0.;
                if (k < k1) {
                    StumpRegs s = load_stump(stumps + k);
                    float f = 0.f;
#pragma unroll
                    for (int j = 0; j < 3; j++) {
                        uint32_t pr = j == 0 ? s.r0 : (j == 1 ? s.r1 : s.r2);
                        float wj = j == 0 ? s.w0 : (j == 1 ? s.w1 : s.w2);
                        if (j == 2 && wj == 0.f) break;
                        int x = pr & 255, y = (pr >> 8) & 255, w = (pr >> 16) & 255, h = pr >> 24;
                        int rs = (int)(win[y * LP + x] - win[y * LP + x + w] - win[(y + h) * LP + x] + win[(y + h) * LP + x + w]);
                        float t = __fmul_rn(wj, __int2float_rn(rs));
                        f = j == 0 ? t : __fadd_rn(f, t);
                    }
                    f = __fmul_rn(f, vnf);
                    leaf = (double)(f < s.thr ? s.left : s.right);
                }
                if (order_free) tmp = __dadd_rn(tmp, leaf);       // per-lane partial, reduced below
                else
                    for (int j = 0; j < 32; j++) tmp = __dadd_rn(tmp, __shfl_sync(0xffffffffu, leaf, j));   // in XML order
            }
            if (order_free)
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) tmp = __dadd_rn(tmp, __shfl_xor_sync(0xffffffffu, tmp, d));
            if (tmp < (double)meta->stage_thr[st]) { code = -st; break; }
        }
        if (lane == 0) {
            if (depth) depth[L.wofs + iy * L.nx + ix] = (int16_t)code;
            if (code == NV_DEPTH_PASS) {
                int pos = atomicAdd(&counters[1], 1);
                if (pos < cand_cap) cand[pos] = q.x;
                else counters[2] = 1;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// k_cascade_tail_fast: k_cascade_tail for cascades with the exactness certificates.  One warp per window, one lane per
// weak classifier of the stage, records prefetched one round ahead, integer feature arithmetic, the stage sum as
// base + sum of (left - right) over the lanes below threshold (DFMA, see add_if_lt) reduced by shuffles.
// ------------------------------------------------------------------------------------------------
// -DNV_TAIL_TRACE: per-phase clock64 sums of the windows that pass every stage (tools/tail_trace.py); compiles out otherwise
#ifdef NV_TAIL_TRACE
__device__ long long g_tail_trace[64 * 16];
__device__ int g_tail_trace_n;
extern "C" __attribute__((visibility("default"))) int nv_debug_tail_trace(long long *out, int cap)
{
    int n = 0;
    cudaMemcpyFromSymbol(&n, g_tail_trace_n, sizeof n);
    cudaMemcpyFromSymbol(out, g_tail_trace, sizeof(long long) * 16 * (n < cap ? n : cap));
    int z = 0;
    cudaMemcpyToSymbol(g_tail_trace_n, &z, sizeof z);
    return n;
}
__device__ __forceinline__ long long clk_after(uint32_t dep)
{
    long long t;
    asm volatile("mov.u64 %0, %%clock64;" : "=l"(t) : "r"(dep));
    return t;
}
#endif
// A warp copies the (wh + 1) x LP integral patch of one window into its shared-memory slot: every lane busy (element
// lane + 32 k; row and column carried along, no division in the loop), four loads in flight per lane.  (Lane per column, row by
// row — 21 of 32 lanes, one load in flight — was 14 % of k_cascade_tail_fast's instructions and 28 % of its stall samples on
// config 3.)
__device__ __forceinline__ void copy_patch(uint32_t *win, const uint32_t *__restrict__ wb, int pitch, int ystep, int iplane, int LP,
                                           int npatch, int lane)
{
    int r = lane / LP, c = lane - r * LP;
    const int dr = 32 / LP, dc = 32 - dr * LP;
    for (int idx = lane; idx < npatch; idx += 128) {
        uint32_t v[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
            if (idx + 32 * u < npatch) v[u] = __ldg(wb + r * pitch + (ystep == 2 ? (c & 1) * iplane + (c >> 1) : c));
            c += dc; r += dr;
            if (c >= LP) { c -= LP; r++; }
        }
#pragma unroll
        for (int u = 0; u < 4; u++)
            if (idx + 32 * u < npatch) win[idx + 32 * u] = v[u];
    }
}

struct TailRec { uint4 a, b, c; };
__device__ __forceinline__ TailRec load_tail(const TailStump *__restrict__ t, int k)
{
    const uint4 *p = reinterpret_cast<const uint4 *>(t + k);
    return TailRec{__ldg(p), __ldg(p + 1), __ldg(p + 2)};
}

__global__ void __launch_bounds__(256)
k_cascade_tail_fast(const PlanDev *__restrict__ plan, const DevCascade *__restrict__ meta, const TailStump *__restrict__ ts,
                    const double *__restrict__ tbase, const uint32_t *__restrict__ sum, const uint2 *__restrict__ tail,
                    int *__restrict__ counters, uint32_t *__restrict__ cand, int cand_cap, int16_t *__restrict__ depth,
                    int stage_begin, int stage_end, uint2 *__restrict__ deep, int deep_cap)
{
    extern __shared__ uint32_t s_win[];                          // 8 warps x (win_h+1) x (win_w+1) words
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // stages [stage_begin, stage_end); a window that gets through them with stages left goes to the `deep` queue
    // (counters[6]) for k_cascade_tail_block.  deep == nullptr: the deep queue is the free part of `tail` itself, behind
    // its n entries (large plans: n is a small fraction of the queue).
    const int n = counters[3], nstages = stage_end, nstumps = meta->nstumps;
    const bool last = stage_end == meta->nstages;
    if (!deep) { deep = const_cast<uint2 *>(tail) + n; deep_cap -= n; }
    const int ww = plan->win_w, wh = plan->win_h, LP = ww + 1, npatch = (wh + 1) * LP;
    uint32_t *win = s_win + warp * npatch;
    const uint32_t wsa = smem_u32(win);
    for (;;) {                                                   // windows are handed out one at a time: depths are very uneven
#ifdef NV_TAIL_TRACE
        long long acc_wait = 0, acc_lds = 0, acc_fp = 0, acc_red = 0, acc_thr = 0, acc_top = 0; int nrounds = 0, nst = 0;
        long long t_begin = clk_after(0);
#endif
        int e = 0;
        if (lane == 0) e = atomicAdd(&counters[5], 1);
        e = __shfl_sync(0xffffffffu, e, 0);
        if (e >= n) break;
        uint2 q = tail[e];
        int l = q.x >> 26, iy = (q.x >> 13) & 8191, ix = q.x & 8191;
        float vnf = __uint_as_float(q.y);
        const LevelDesc &L = plan->lv[l];
        const uint32_t *wb = sum + L.iofs + (size_t)iy * L.ystep * L.ipitch + ix;
        int k0 = meta->stage_first[stage_begin];
        TailRec rec = load_tail(ts, min(k0 + lane, nstumps - 1));
        __syncwarp();
        copy_patch(win, wb, L.ipitch, L.ystep, L.iplane, LP, npatch, lane);       // private copy of the window's integral patch
        __syncwarp();
#ifdef NV_TAIL_TRACE
        long long t_copied = clk_after((uint32_t)win[0]);
        long long tp = t_copied;
#endif
        int code = NV_DEPTH_PASS;
        for (int st = stage_begin; st < nstages; st++) {
            int k1 = meta->stage_first[st + 1];
            double tmp = 0.;
#ifdef NV_TAIL_TRACE
            { long long t = clk_after((uint32_t)k1); acc_top += t - tp; tp = t; nst++; }
#endif
            for (int kb = k0; kb < k1; kb += 32) {               // 32 weak classifiers per round, one per lane
                TailRec cur = rec;
                int nk = (kb + 32 < k1 ? kb + 32 : k1) + lane;   // next round: same stage, or the head of the next one
                rec = load_tail(ts, min(nk, nstumps - 1));
#ifdef NV_TAIL_TRACE
                { long long t = clk_after(cur.a.x ^ cur.b.x ^ cur.c.y); acc_wait += t - tp; tp = t; nrounds++; }
                int r_dep = 0;
#endif
                if (kb + lane < k1) {
#define TW(o) lds_u32(wsa + (o))
                    int nr0 = (int)(TW(cur.a.x >> 16) + TW(cur.a.y & 0xffffu) - TW(cur.a.x & 0xffffu) - TW(cur.a.y >> 16));
                    int r1 = (int)(TW(cur.a.z & 0xffffu) - TW(cur.a.z >> 16) - TW(cur.a.w & 0xffffu) + TW(cur.a.w >> 16));
                    int w12 = (int)cur.b.w;
                    int r = (int)(short)(w12 & 0xffff) * r1 + nr0;
                    if (w12 >> 16) {
                        int r2 = (int)(TW(cur.b.x & 0xffffu) - TW(cur.b.x >> 16) - TW(cur.b.y & 0xffffu) + TW(cur.b.y >> 16));
                        r += (w12 >> 16) * r2;
                    }
#undef TW
#ifdef NV_TAIL_TRACE
                    r_dep = r;
                    { long long t = clk_after((uint32_t)r_dep); acc_lds += t - tp; tp = t; }
#endif
                    add_if_lt(tmp, __fmul_rn(__int2float_rn(r), vnf), __uint_as_float(cur.b.z),
                              __hiloint2double((int)cur.c.y, (int)cur.c.x));
                }
#ifdef NV_TAIL_TRACE
                { long long t = clk_after((uint32_t)__double2hiint(tmp)); acc_fp += t - tp; tp = t; }
#endif
            }
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) tmp = __dadd_rn(tmp, __shfl_xor_sync(0xffffffffu, tmp, d));
            k0 = k1;
#ifdef NV_TAIL_TRACE
            { long long t = clk_after((uint32_t)__double2hiint(tmp)); acc_red += t - tp; tp = t; }
            bool failed = __dadd_rn(tbase[st], tmp) < (double)meta->stage_thr[st];
            { long long t = clk_after((uint32_t)failed); acc_thr += t - tp; tp = t; }
            if (failed) { code = -st; break; }
#else
            if (__dadd_rn(tbase[st], tmp) < (double)meta->stage_thr[st]) { code = -st; break; }
#endif
        }
#ifdef NV_TAIL_TRACE
        if (lane == 0 && code == NV_DEPTH_PASS) {
            int slot = atomicAdd(&g_tail_trace_n, 1);
            if (slot < 64) {
                long long *o = g_tail_trace + slot * 16;
                o[0] = tp - t_begin; o[1] = t_copied - t_begin; o[2] = acc_top; o[3] = acc_wait; o[4] = acc_lds; o[5] = acc_fp;
                o[6] = acc_red; o[7] = acc_thr; o[8] = nrounds; o[9] = nst;
            }
        }
#endif
        if (lane == 0) {
            if (depth && (last || code != NV_DEPTH_PASS)) depth[L.wofs + iy * L.nx + ix] = (int16_t)code;
            if (code == NV_DEPTH_PASS && last) {
                int pos = atomicAdd(&counters[1], 1);
                if (pos < cand_cap) cand[pos] = q.x;
                else counters[2] = 1;
            } else if (code == NV_DEPTH_PASS) {
                int pos = atomicAdd(&counters[6], 1);
                if (pos < deep_cap) deep[pos] = q;
                else counters[2] = 1;
            }
        }
    }
}

// k_cascade_tail_tab: k_cascade_tail_fast with the weak classifiers of its stage range IN SHARED MEMORY.  The clock64
// timeline of a full-depth window (profiles/r1_v5_summary.md) put a third of every round of 32 classifiers into waiting
// for the lanes' 48-byte records from L2 — a round is shorter than the L2 round trip, so a one-round prefetch cannot
// hide it — and that chain (61 rounds for stages 10..21 of frontalface_alt) is what the launch takes whatever the frame
// holds.  Here a block copies the records of stages [stage_begin, nstages) once (40 bytes each as three arrays: lane k
// reads element k, no bank conflicts; 70 KB for stages 10..21, 85 KB from stage 1), a lane takes TWO classifiers per round
// (half the rounds, the two evaluations overlap), and the stage bounds / thresholds / base sums sit in shared memory
// too.  Fewer, fatter blocks: as many per SM as the table allows, persistent over the window queue.  Same certificates,
// same arithmetic, same results as k_cascade_tail_fast; used when the table fits (launch_cascade_tail_tab).
// BATCH: the queue holds the windows of a batch of images, (image << 14) | dense window index (k_stage0_rows_p<true>); the
// image's integrals lie at image * integ_stride, its candidates go to its own segment cand + image * cand_stride with the
// count in its own counter block (counters + 16 * (1 + image)).  Queue count and ticket stay in counters[3] / [5].
template <int NWARP, bool BATCH>
__global__ void __launch_bounds__(32 * NWARP)
k_cascade_tail_tab(const PlanDev *__restrict__ plan, const DevCascade *__restrict__ meta, const TailStump *__restrict__ ts,
                   const double *__restrict__ tbase, const uint32_t *__restrict__ sum, const uint2 *__restrict__ tail,
                   int *__restrict__ counters, uint32_t *__restrict__ cand, int cand_cap, int16_t *__restrict__ depth,
                   int stage_begin, int stage_end, uint2 *__restrict__ deep, int deep_cap, size_t integ_stride = 0, int cand_stride = 0)
{
    extern __shared__ __align__(16) uint32_t s_tab[];            // A[nt] uint4 | B[nt] uint4 | C[nt] double | NWARP patches
    __shared__ int s_first[NV_MAX_STAGES + 1];
    __shared__ float s_thr[NV_MAX_STAGES];
    __shared__ double s_base[NV_MAX_STAGES];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n = counters[3], nstages = stage_end;
    if (n == 0) return;
    const bool last = stage_end == meta->nstages;
    if (!deep) { deep = const_cast<uint2 *>(tail) + n; deep_cap -= n; }
    const int kt0 = meta->stage_first[stage_begin], nt = meta->stage_first[stage_end] - kt0;
    uint4 *sA = reinterpret_cast<uint4 *>(s_tab), *sB = sA + nt;
    double *sC = reinterpret_cast<double *>(sB + nt);
    const int ww = plan->win_w, wh = plan->win_h, LP = ww + 1, npatch = (wh + 1) * LP;
    uint32_t *win = reinterpret_cast<uint32_t *>(sC + nt) + warp * npatch;
    for (int i0 = tid; i0 < nt; i0 += 4 * 32 * NWARP) {          // four records per thread in flight (a thread copies ~9 of them)
        uint4 ra[4], rb[4], rc[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int i = i0 + u * 32 * NWARP;
            if (i < nt) {
                const uint4 *p = reinterpret_cast<const uint4 *>(ts + kt0 + i);
                ra[u] = __ldg(p); rb[u] = __ldg(p + 1); rc[u] = __ldg(p + 2);
            }
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int i = i0 + u * 32 * NWARP;
            if (i < nt) { sA[i] = ra[u]; sB[i] = rb[u]; sC[i] = __hiloint2double((int)rc[u].y, (int)rc[u].x); }
        }
    }
    for (int i = tid; i <= meta->nstages; i += 32 * NWARP) s_first[i] = meta->stage_first[i] - kt0;
    for (int i = tid; i < meta->nstages; i += 32 * NWARP) { s_thr[i] = meta->stage_thr[i]; s_base[i] = tbase[i]; }
    __syncthreads();
    const uint32_t wsa = smem_u32(win);
    for (;;) {                                                   // windows are handed out one at a time: depths are very uneven
        int e = 0;
        if (lane == 0) e = atomicAdd(&counters[5], 1);
        e = __shfl_sync(0xffffffffu, e, 0);
        if (e >= n) break;
        const uint2 q = tail[e];
        int l, iy, ix;
        uint32_t id = q.x;
        const uint32_t *isum = sum;
        int *icnt = counters;
        uint32_t *icand = cand;
        int icap = cand_cap;
        if (BATCH) {
            const int img = q.x >> 14, w = q.x & 16383;
            l = 0;
            while (l + 1 < plan->nlevels && plan->lv[l + 1].wofs <= w) l++;
            const int r = w - plan->lv[l].wofs;
            iy = r / plan->lv[l].nx; ix = r - iy * plan->lv[l].nx;
            id = ((uint32_t)l << 26) | ((uint32_t)iy << 13) | (uint32_t)ix;
            isum = sum + img * integ_stride; icnt = counters + 16 * (1 + img);
            icand = cand + img * (size_t)cand_stride; icap = cand_stride;
        } else {
            l = q.x >> 26; iy = (q.x >> 13) & 8191; ix = q.x & 8191;
        }
        const float vnf = __uint_as_float(q.y);
        const LevelDesc &L = plan->lv[l];
        const int pitch = L.ipitch;
        const uint32_t *wb = isum + L.iofs + (size_t)iy * L.ystep * pitch + ix;
        __syncwarp();                                            // the previous window's reads of the patch are done
        copy_patch(win, wb, pitch, L.ystep, L.iplane, LP, npatch, lane);         // private copy of the window's integral patch
        __syncwarp();
        int code = NV_DEPTH_PASS;
        for (int st = stage_begin; st < nstages; st++) {
            const int k0 = s_first[st], k1 = s_first[st + 1];
            double tmp0 = 0., tmp1 = 0.;
            for (int kb = k0 + lane; kb < k1; kb += 64) {        // 64 weak classifiers per round, two per lane
#define TW(o) lds_u32(wsa + (o))
#define TAIL_EVAL(K, ACC)                                                                                              \
                {                                                                                                      \
                    const uint4 a = sA[K], b = sB[K];                                                                  \
                    const int nr0 = (int)(TW(a.x >> 16) + TW(a.y & 0xffffu) - TW(a.x & 0xffffu) - TW(a.y >> 16));      \
                    const int r1 = (int)(TW(a.z & 0xffffu) - TW(a.z >> 16) - TW(a.w & 0xffffu) + TW(a.w >> 16));      \
                    const int w12 = (int)b.w;                                                                          \
                    int r = (int)(short)(w12 & 0xffff) * r1 + nr0;                                                     \
                    if (w12 >> 16) {                                                                                   \
                        const int r2 = (int)(TW(b.x & 0xffffu) - TW(b.x >> 16) - TW(b.y & 0xffffu) + TW(b.y >> 16));  \
                        r += (w12 >> 16) * r2;                                                                         \
                    }                                                                                                  \
                    add_if_lt(ACC, __fmul_rn(__int2float_rn(r), vnf), __uint_as_float(b.z), sC[K]);                    \
                }
                TAIL_EVAL(kb, tmp0)
                if (kb + 32 < k1) TAIL_EVAL(kb + 32, tmp1)
#undef TAIL_EVAL
#undef TW
            }
            double tmp = __dadd_rn(tmp0, tmp1);
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) tmp = __dadd_rn(tmp, __shfl_xor_sync(0xffffffffu, tmp, d));
            if (__dadd_rn(s_base[st], tmp) < (double)s_thr[st]) { code = -st; break; }
        }
        if (lane == 0) {
            if (depth && (last || code != NV_DEPTH_PASS)) depth[L.wofs + iy * L.nx + ix] = (int16_t)code;
            if (code == NV_DEPTH_PASS && last) {
                const int pos = atomicAdd(&icnt[1], 1);
                if (pos < icap) icand[pos] = id;
                else icnt[2] = 1;
            } else if (code == NV_DEPTH_PASS) {
                const int pos = atomicAdd(&counters[6], 1);
                if (pos < deep_cap) deep[pos] = q;
                else counters[2] = 1;
            }
        }
    }
}

// The deep stages (80 .. 213 weak classifiers each in frontalface_alt) with a whole BLOCK per window: one classifier per
// thread, so a stage is one round (two for the last ones) instead of three to seven, and the stage sum is combined through
// shared memory with one barrier per stage.  A window that passes all 22 stages costs ~12 short rounds here against ~55 in
// the warp-per-window kernel: that chain was the floor of every call (41-46 us, profiles/r1_v5_summary.md).  Needs the same
// order-free certificate as k_cascade_tail_fast (the partial sums are added in another order).
__global__ void __launch_bounds__(256)
k_cascade_tail_block(const PlanDev *__restrict__ plan, const DevCascade *__restrict__ meta, const TailStump *__restrict__ ts,
                     const double *__restrict__ tbase, const uint32_t *__restrict__ sum, const uint2 *__restrict__ queue,
                     int *__restrict__ counters, int cin, uint32_t *__restrict__ cand, int cand_cap, int16_t *__restrict__ depth,
                     int stage_begin, int skip_counter)
{
    if (skip_counter >= 0) queue += counters[skip_counter];      // the deep queue sits behind the tail queue's entries
    __shared__ uint32_t s_patch[33 * 33];
    __shared__ double s_part[2][8];
    __shared__ int s_first[NV_MAX_STAGES + 1];
    __shared__ float s_thr[NV_MAX_STAGES];
    __shared__ double s_base[NV_MAX_STAGES];
    __shared__ int s_e;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n = counters[cin], nstages = meta->nstages, nstumps = meta->nstumps;
    if (n == 0) return;
    const int ww = plan->win_w, wh = plan->win_h, LP = ww + 1, npatch = (wh + 1) * LP;
    for (int i = tid; i <= nstages; i += 256) s_first[i] = meta->stage_first[i];
    for (int i = tid; i < nstages; i += 256) { s_thr[i] = meta->stage_thr[i]; s_base[i] = tbase[i]; }
    const uint32_t wsa = smem_u32(s_patch);
    for (;;) {
        __syncthreads();                                         // the previous window is done with s_patch and s_e
        if (tid == 0) s_e = atomicAdd(&counters[7], 1);
        __syncthreads();
        const int e = s_e;
        if (e >= n) break;
        const uint2 q = queue[e];
        const int l = q.x >> 26, iy = (q.x >> 13) & 8191, ix = q.x & 8191;
        const float vnf = __uint_as_float(q.y);
        const LevelDesc &L = plan->lv[l];
        const uint32_t *wb = sum + L.iofs + (size_t)iy * L.ystep * L.ipitch + ix;
        int k0 = s_first[stage_begin];
        TailRec rec = load_tail(ts, min(k0 + tid, nstumps - 1));
        for (int idx = tid; idx < npatch; idx += 256) {          // the window's integral patch
            const int r = idx / LP, c = idx - r * LP;
            const int pc = L.ystep == 2 ? (c & 1) * L.iplane + (c >> 1) : c;
            s_patch[idx] = __ldg(wb + (size_t)r * L.ipitch + pc);
        }
        __syncthreads();
        int code = NV_DEPTH_PASS;
        for (int st = stage_begin; st < nstages; st++) {
            const int k1 = s_first[st + 1];
            double tmp = 0.;
            for (int kb = k0; kb < k1; kb += 256) {
                const TailRec cur = rec;
                const int nk = (kb + 256 < k1 ? kb + 256 : k1) + tid;           // next round: same stage, or the head of the next one
                rec = load_tail(ts, min(nk, nstumps - 1));
                if (kb + tid < k1) {
#define TW(o) lds_u32(wsa + (o))
                    const int nr0 = (int)(TW(cur.a.x >> 16) + TW(cur.a.y & 0xffffu) - TW(cur.a.x & 0xffffu) - TW(cur.a.y >> 16));
                    const int r1 = (int)(TW(cur.a.z & 0xffffu) - TW(cur.a.z >> 16) - TW(cur.a.w & 0xffffu) + TW(cur.a.w >> 16));
                    const int w12 = (int)cur.b.w;
                    int r = (int)(short)(w12 & 0xffff) * r1 + nr0;
                    if (w12 >> 16) {
                        const int r2 = (int)(TW(cur.b.x & 0xffffu) - TW(cur.b.x >> 16) - TW(cur.b.y & 0xffffu) + TW(cur.b.y >> 16));
                        r += (w12 >> 16) * r2;
                    }
#undef TW
                    add_if_lt(tmp, __fmul_rn(__int2float_rn(r), vnf), __uint_as_float(cur.b.z), __hiloint2double((int)cur.c.y, (int)cur.c.x));
                }
            }
            // warps that hold no classifier of this stage contribute an exact 0
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) tmp = __dadd_rn(tmp, __shfl_xor_sync(0xffffffffu, tmp, d));
            if (lane == 0) s_part[st & 1][warp] = tmp;
            __syncthreads();
            double total = s_base[st];
#pragma unroll
            for (int w = 0; w < 8; w++) total = __dadd_rn(total, s_part[st & 1][w]);
            k0 = k1;
            if (total < (double)s_thr[st]) { code = -st; break; }                  // block-uniform: every thread adds the same values
        }
        if (tid == 0) {
            if (depth) depth[L.wofs + iy * L.nx + ix] = (int16_t)code;
            if (code == NV_DEPTH_PASS) {
                const int pos = atomicAdd(&counters[1], 1);
                if (pos < cand_cap) cand[pos] = q.x;
                else counters[2] = 1;
            }
        }
    }
}

// host: the TailStump table and the certificate over every stage (same conditions as fill_bulk_stumps' FAST variant)
void build_tail_stumps(nv_cascade *c)
{
    const DevCascade &m = c->meta;
    bool fast = c->h.order_free != 0 && m.win_w <= 32 && m.win_h <= 32;
    for (int k = 0; k < m.nstumps && fast; k++) {
        const DevStump &d = c->stumps[k];
        double bound = 0;
        for (int j = 0; j < 3; j++) {
            if (d.w[j] != rintf(d.w[j]) || fabsf(d.w[j]) > 4096.f) fast = false;
            bound += fabs((double)d.w[j]) * ((d.r[j] >> 16) & 255) * (d.r[j] >> 24) * 255.0;
        }
        if (bound >= 16777216.0 || d.w[0] != -1.f) fast = false;
    }
    c->tail_fast = fast ? 1 : 0;
    if (!fast) return;
    const int LP = m.win_w + 1;
    c->tail_stumps.clear(); c->tail_base.assign(m.nstages, 0.0);
    for (int s = 0; s < m.nstages; s++) {
        double rsum = 0;
        for (int grp = 0; grp < 2; grp++)
            for (int k = m.stage_first[s]; k < m.stage_first[s + 1]; k++) {
                const DevStump &d = c->stumps[k];
                if ((d.w[2] != 0.f) != (grp == 1)) continue;
                TailStump t;
                memset(&t, 0, sizeof t);
                for (int j = 0; j < 3; j++) {
                    uint32_t r = (j < 2 || d.w[2] != 0.f) ? d.r[j] : d.r[0];
                    int x = r & 255, y = (r >> 8) & 255, w = (r >> 16) & 255, h = r >> 24;
                    t.o[4 * j + 0] = (uint16_t)(4 * (y * LP + x));       t.o[4 * j + 1] = (uint16_t)(4 * (y * LP + x + w));
                    t.o[4 * j + 2] = (uint16_t)(4 * ((y + h) * LP + x)); t.o[4 * j + 3] = (uint16_t)(4 * ((y + h) * LP + x + w));
                }
                t.thr = d.thr; t.w1 = (int16_t)d.w[1]; t.w2 = (int16_t)d.w[2];
                t.d128 = 128.0 * ((double)d.left - (double)d.right);
                rsum += (double)d.right;
                c->tail_stumps.push_back(t);
            }
        c->tail_base[s] = rsum;
    }
}

// host: bulk-stage weak classifiers with shared-memory corner BYTE offsets for one ystep class, plus the
// certificates of the FAST variant:
//   order-free — cascade_xml.cpp proves that no addition of a stage's leaves can round in double, so any order and the
//     "sum of right leaves + (left - right) of the classifiers below threshold" form give the reference's stage sum
//     (every partial sum is a sum of one leaf per classifier, a multiple of the smallest leaf ulp below 2^52 ulps);
//   integer features — the first rect of every bulk-stage feature weighs -1, the other weights are integers and
//     sum_j |w_j| * area_j * 255 < 2^24, so every float product and sum of the reference's feature evaluation is
//     exact and equals the int32 evaluation w1*r1 (+ w2*r2) - r0.
// FAST order inside a stage: two-rect features whose rects share two corners (one rect is a half of the other),
// other two-rect features, three-rect features.  For the first group r0 = U - V and r1 = U - V' with a common
// difference U of two corner values: six loads instead of eight.  o0 = (p0, p1, p2, p3), o1 = (p4, p5) with
//   U = p0 - p1,  -r0 = (p2 - p3) - U,  r1 = U - p4 + p5
// which covers the four sharing patterns by the choice of p (a, b, c, d = corners of rect 0; a1.. of rect 1):
//   left half  (a = a1, c = c1): p = a, c, b, d, b1, d1        right half  (b = b1, d = d1): p = d, b, c, a, c1, a1
//   top half   (a = a1, b = b1): p = a, b, c, d, c1, d1        bottom half (c = c1, d = d1): p = d, c, b, a, b1, a1
// One stage's weak classifiers in the bulk kernels' form, appended at S[n], O2[n].  FAST: group 0 = six-load two-rect,
// 1 = eight-load two-rect, 2 = three-rect (mid6 / mid = where groups 1 / 2 start); otherwise XML order in one group.
// base = sum of the stage's right leaves.
static void fill_stage_stumps(const nv_cascade *c, int ystep, int cp, int ps, int s, bool fast, BulkStump *S, uint4 *O2, int *n_io,
                              int *mid6, int *mid, double *base)
{
    const DevCascade &m = c->meta;
    auto off = [&](int dx, int dy) { return 4u * (uint32_t)(ystep == 2 ? (dx & 1) * ps + dy * cp + (dx >> 1) : dy * cp + dx); };
    auto f2u = [](float f) { uint32_t u; memcpy(&u, &f, 4); return u; };
    struct Corners {
        uint32_t a, b, c, d;
        bool eq(const Corners &o, int i) const { return i == 0 ? a == o.a : i == 1 ? b == o.b : i == 2 ? c == o.c : d == o.d; }
    };
    auto corners = [&](uint32_t r) {
        int x = r & 255, y = (r >> 8) & 255, w = (r >> 16) & 255, h = r >> 24;
        return Corners{off(x, y), off(x + w, y), off(x, y + h), off(x + w, y + h)};
    };
    // sharing pattern of a two-rect feature: 0 none, 1 left half, 2 right half, 3 top half, 4 bottom half
    auto pattern = [&](const DevStump &d) {
        if (d.w[2] != 0.f) return 0;
        Corners p = corners(d.r[0]), q = corners(d.r[1]);
        bool e[4] = {p.eq(q, 0), p.eq(q, 1), p.eq(q, 2), p.eq(q, 3)};
        if (e[0] && e[2] && !e[1] && !e[3]) return 1;
        if (e[1] && e[3] && !e[0] && !e[2]) return 2;
        if (e[0] && e[1] && !e[2] && !e[3]) return 3;
        if (e[2] && e[3] && !e[0] && !e[1]) return 4;
        return 0;
    };
    int n = *n_io;
    double rsum = 0;
    *mid6 = *mid = n;
    for (int grp = 0; grp < (fast ? 3 : 1); grp++) {
        for (int k = m.stage_first[s]; k < m.stage_first[s + 1]; k++) {
            const DevStump &d = c->stumps[k];
            bool three = d.w[2] != 0.f;
            int pat = pattern(d);
            if (fast && (three ? 2 : (pat ? 0 : 1)) != grp) continue;
            BulkStump &b = S[n];
            Corners p = corners(d.r[0]), q = corners(d.r[1]), t = corners(three ? d.r[2] : d.r[0]);
            b.o0 = make_uint4(p.a, p.b, p.c, p.d); b.o1 = make_uint4(q.a, q.b, q.c, q.d); O2[n] = make_uint4(t.a, t.b, t.c, t.d);
            if (fast && pat == 1) { b.o0 = make_uint4(p.a, p.c, p.b, p.d); b.o1 = make_uint4(q.b, q.d, 0, 0); }
            if (fast && pat == 2) { b.o0 = make_uint4(p.d, p.b, p.c, p.a); b.o1 = make_uint4(q.c, q.a, 0, 0); }
            if (fast && pat == 3) { b.o0 = make_uint4(p.a, p.b, p.c, p.d); b.o1 = make_uint4(q.c, q.d, 0, 0); }
            if (fast && pat == 4) { b.o0 = make_uint4(p.d, p.c, p.b, p.a); b.o1 = make_uint4(q.b, q.a, 0, 0); }
            if (fast) { b.w0 = (uint32_t)(int)d.w[0]; b.w1 = (uint32_t)(int)d.w[1]; b.w2 = (uint32_t)(int)d.w[2]; }
            else { b.w0 = f2u(d.w[0]); b.w1 = f2u(d.w[1]); b.w2 = f2u(d.w[2]); }
            b.thr = f2u(d.thr); b.left = f2u(d.left); b.right = f2u(d.right);
            double dd = 128.0 * ((double)d.left - (double)d.right);          // see add_if_lt
            uint64_t u; memcpy(&u, &dd, 8);
            b.d_lo = (uint32_t)u; b.d_hi = (uint32_t)(u >> 32);
            rsum += (double)d.right;
            n++;
        }
        if (grp == 0 && fast) *mid6 = n;
        if (grp == 1 && fast) *mid = n;
    }
    if (!fast) *mid6 = *mid = *n_io;
    *base = rsum;
    *n_io = n;
}

// exactness certificates of stages [stage_begin, stage_end): order-free stage sums (cascade_xml.cpp) and integer feature
// arithmetic — rect 0 weighs -1, the other weights are small integers and sum |w| * area * 255 < 2^24
static bool stages_are_fast(const nv_cascade *c, int stage_begin, int stage_end)
{
    const DevCascade &m = c->meta;
    bool fast = c->h.order_free != 0;
    for (int k = m.stage_first[stage_begin]; k < m.stage_first[stage_end] && fast; k++) {
        const DevStump &d = c->stumps[k];
        double bound = 0;
        for (int j = 0; j < 3; j++) {
            if (d.w[j] != rintf(d.w[j]) || fabsf(d.w[j]) > 4096.f) fast = false;
            bound += fabs((double)d.w[j]) * ((d.r[j] >> 16) & 255) * (d.r[j] >> 24) * 255.0;
        }
        if (bound >= 16777216.0 || d.w[0] != -1.f) fast = false;
    }
    return fast;
}

void fill_bulk_stumps(const nv_cascade *c, int ystep, int cp, int ps, int stage_begin, int stage_end, TileParams *tp)
{
    const DevCascade &m = c->meta;
    tp->stage_begin = stage_begin;
    tp->stage_end = stage_end;
    tp->final_stage = stage_end == m.nstages;
    const bool fast = stages_are_fast(c, stage_begin, stage_end);
    tp->fast = fast ? 1 : 0;
    int n = 0;
    for (int s = stage_begin; s < stage_end; s++) {
        const int si = s - stage_begin;
        tp->stage_first[si] = n;
        tp->stage_thr[si] = m.stage_thr[s];
        fill_stage_stumps(c, ystep, cp, ps, s, fast, tp->s, tp->o2, &n, &tp->stage_mid6[si], &tp->stage_mid[si], &tp->stage_base[si]);
    }
    tp->stage_first[stage_end - stage_begin] = n;
}

// stage 0 in the tile layout of one ystep class; false when stage 0 lacks the exactness certificates or is too wide
bool fill_stage0_tile_params(const nv_cascade *c, int ystep, int cp, int rt, int ps, int kskew, Stage0TileParams *sp)
{
    const DevCascade &m = c->meta;
    const int n0 = m.stage_first[1];
    if (n0 > NV_S0T_MAX_STUMPS || n0 < 1 || !stages_are_fast(c, 0, 1)) return false;
    int n = 0;
    sp->stage_first[0] = 0;
    sp->stage_thr[0] = m.stage_thr[0];
    fill_stage_stumps(c, ystep, cp, ps, 0, true, sp->s, sp->o2, &n, &sp->stage_mid6[0], &sp->stage_mid[0], &sp->stage_base[0]);
    sp->stage_first[1] = n;
    auto off = [&](int dx, int dy) { return 4u * (uint32_t)(ystep == 2 ? (dx & 1) * ps + dy * cp + (dx >> 1) : dy * cp + dx); };
    sp->var = make_uint4(off(1, 1), off(m.win_w - 1, 1), off(1, m.win_h - 1), off(m.win_w - 1, m.win_h - 1));
    sp->win_w = m.win_w; sp->win_h = m.win_h;
    sp->cp = cp; sp->rt = rt; sp->ps = ps; sp->kskew = kskew;
    return true;
}

// ------------------------------------------------------------------------------------------------
cudaError_t launch_queue_stages(const PlanDev *plan, const DevCascade *meta, const DevStump *stumps, const uint32_t *sum,
                                const uint2 *queue, int *counters, uint32_t *cand, int cand_cap, int16_t *depth,
                                int nblocks, cudaStream_t st)
{
    k_queue_stages<<<nblocks, 256, 0, st>>>(plan, meta, stumps, sum, queue, counters, cand, cand_cap, depth);
    return cudaGetLastError();
}

cudaError_t launch_stage0_rows(const PlanDev *plan, int total_rows, const DevCascade *meta, const DevStump *stumps,
                               const uint32_t *sum, const uint32_t *sq, float *vnf, uint32_t *bits_alive, int *counters,
                               int16_t *depth, cudaStream_t st)
{
    k_stage0_rows<<<(total_rows + 7) / 8, 256, 0, st>>>(plan, total_rows, meta, stumps, sum, sq, vnf, bits_alive, counters, depth);
    return cudaGetLastError();
}

// cidx: the counter the queue positions are allocated from — 4 for the generic queue kernels (they take their count
// from counters[0]), 3 when the queue feeds k_cascade_tail_fast (its count)
cudaError_t launch_alive_to_queue(const PlanDev *plan, int total_rows, const float *vnf, const uint32_t *bits_alive,
                                  uint2 *queue, int *counters, int queue_cap, cudaStream_t st, int cidx)
{
    k_alive_to_queue<<<(total_rows + 7) / 8, 256, 0, st>>>(plan, total_rows, vnf, bits_alive, queue, counters, queue_cap, cidx);
    return cudaGetLastError();
}

// The dynamic shared-memory limit is an attribute of a device's copy of a kernel: raised once per (kernel, device).
static cudaError_t raise_smem_limit(const void *kernel, int bytes)
{
    static std::mutex mu;
    static std::set<std::pair<const void *, int>> done;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lk(mu);
    if (done.count({kernel, dev})) return cudaSuccess;
    if ((e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes)) == cudaSuccess) done.insert({kernel, dev});
    return e;
}

cudaError_t launch_stage0_tiles(const Stage0TileParams &sp, int ystep, int ntiles, cudaStream_t st)
{
    const auto kernel = ystep == 2 ? k_stage0_tiles<2> : k_stage0_tiles<1>;
    cudaError_t e = raise_smem_limit((const void *)kernel, 160 * 1024);
    if (e != cudaSuccess) return e;
    kernel<<<ntiles, 256, (size_t)ystep * sp.ps * sizeof(uint32_t), st>>>(sp);
    return cudaGetLastError();
}

cudaError_t launch_stage0_chain(const PlanDev &plan, const uint32_t *bits_fail, const uint32_t *bits_okv,
                                uint32_t *bits_alive, int *counters, int16_t *depth, cudaStream_t st)
{
    ChainParams cp;
    for (int l = 0; l < plan.nlevels; l++) {
        const LevelDesc &L = plan.lv[l];
        cp.a[l] = make_int4(L.row0, L.nxw, L.nx, L.bofs); cp.wofs[l] = L.wofs;
    }
    cp.nlevels = plan.nlevels; cp.total_rows = plan.total_rows;
    cp.bits_fail = bits_fail; cp.bits_okv = bits_okv; cp.bits_alive = bits_alive; cp.counters = counters; cp.depth = depth;
    k_stage0_chain<<<(plan.total_rows + 7) / 8, 256, 0, st>>>(cp);
    return cudaGetLastError();
}

// the bulk stages of the ystep-2 levels: NV_CTX x NV_CTY-window tiles, two column planes each
cudaError_t launch_cascade_classes(const TileParams &tp, int ntiles, cudaStream_t st)
{
    const auto kernel = tp.fast ? k_cascade_classes<2, true> : k_cascade_classes<2, false>;
    cudaError_t e = raise_smem_limit((const void *)kernel, 160 * 1024);
    if (e != cudaSuccess) return e;
    kernel<<<ntiles, 256, 2 * (size_t)tp.ps * sizeof(uint32_t), st>>>(tp);
    return cudaGetLastError();
}

// the bulk stages of the ystep-1 levels: NV_WTX x NV_WTY-window tiles, eight warps
cudaError_t launch_cascade_wide(const TileParams &tp, int ntiles, cudaStream_t st)
{
    const auto kernel = tp.fast ? k_cascade_wide<1, true, NV_WTX, NV_WTY, 8> : k_cascade_wide<1, false, NV_WTX, NV_WTY, 8>;
    cudaError_t e = raise_smem_limit((const void *)kernel, 160 * 1024);
    if (e != cudaSuccess) return e;
    kernel<<<ntiles, 32 * 8, (size_t)tp.ps * sizeof(uint32_t), st>>>(tp);
    return cudaGetLastError();
}

cudaError_t launch_cascade_tail(const PlanDev *plan, const DevCascade *meta, const DevStump *stumps, const uint32_t *sum,
                                const uint2 *tail, int *counters, uint32_t *cand, int cand_cap, int16_t *depth,
                                int stage_begin, int order_free, int nblocks, cudaStream_t st, int smem_bytes)
{
    (void)nblocks;
    k_cascade_tail<<<148 * 8, 256, smem_bytes, st>>>(plan, meta, stumps, sum, tail, counters, cand, cand_cap, depth, stage_begin,
                                                     order_free);
    return cudaGetLastError();
}

cudaError_t launch_cascade_tail_block(const PlanDev *plan, const DevCascade *meta, const TailStump *tstumps, const double *tbase,
                                      const uint32_t *sum, const uint2 *queue, int *counters, int cin, uint32_t *cand, int cand_cap,
                                      int16_t *depth, int stage_begin, int skip_counter, cudaStream_t st)
{
    k_cascade_tail_block<<<148 * 4, 256, 0, st>>>(plan, meta, tstumps, tbase, sum, queue, counters, cin, cand, cand_cap, depth, stage_begin,
                                                 skip_counter);
    return cudaGetLastError();
}

cudaError_t launch_cascade_tail_fast(const PlanDev *plan, const DevCascade *meta, const TailStump *tstumps, const double *tbase,
                                     const uint32_t *sum, const uint2 *tail, int *counters, uint32_t *cand, int cand_cap,
                                     int16_t *depth, int stage_begin, int stage_end, uint2 *deep, int deep_cap, cudaStream_t st,
                                     int smem_bytes)
{
#ifndef NV_TAIL_THREADS
#define NV_TAIL_THREADS 256
#endif
    // smem_bytes is sized for eight warps (one patch per warp)
    k_cascade_tail_fast<<<148 * 8 * (256 / NV_TAIL_THREADS), NV_TAIL_THREADS, smem_bytes / (256 / NV_TAIL_THREADS), st>>>(
        plan, meta, tstumps, tbase, sum, tail, counters, cand, cand_cap, depth, stage_begin, stage_end, deep, deep_cap);
    return cudaGetLastError();
}

// Shared-memory bytes of k_cascade_tail_tab for the stage range [stage_begin, nstages) of a cascade, and the launch.
// Returns cudaErrorInvalidConfiguration when the table does not fit: the caller falls back to k_cascade_tail_fast.
#ifndef NV_TAILTAB_WARPS
#define NV_TAILTAB_WARPS 8
#endif
size_t tail_tab_smem(const DevCascade &m, int stage_begin, int stage_end)
{
    const size_t nt = (size_t)(m.stage_first[stage_end] - m.stage_first[stage_begin]);
    return nt * 40 + (size_t)NV_TAILTAB_WARPS * (m.win_w + 1) * (m.win_h + 1) * 4;
}

template <bool BATCH>
static cudaError_t launch_tail_tab_t(const PlanDev *plan, const DevCascade *meta, const DevCascade &hmeta, const TailStump *tstumps,
                                     const double *tbase, const uint32_t *sum, const uint2 *tail, int *counters, uint32_t *cand,
                                     int cand_cap, int16_t *depth, int stage_begin, int stage_end, uint2 *deep, int deep_cap,
                                     cudaStream_t st, size_t integ_stride, int cand_stride)
{
    const size_t smem = tail_tab_smem(hmeta, stage_begin, stage_end);
    if (smem > NV_TAILTAB_MAX_SMEM) return cudaErrorInvalidConfiguration;
    cudaError_t e = raise_smem_limit((const void *)k_cascade_tail_tab<NV_TAILTAB_WARPS, BATCH>, (int)NV_TAILTAB_MAX_SMEM);
    if (e != cudaSuccess) return e;
    int per_sm = (int)((227 * 1024) / (smem + 2048));            // static tables + the per-block reserve
    per_sm = per_sm < 1 ? 1 : per_sm > 8 ? 8 : per_sm;
    // (fewer blocks when the queue is short — every block copies the table — was measured: no gain down to one block per 32
    // windows of the plan, slower below)
    k_cascade_tail_tab<NV_TAILTAB_WARPS, BATCH><<<148 * per_sm, 32 * NV_TAILTAB_WARPS, smem, st>>>(
        plan, meta, tstumps, tbase, sum, tail, counters, cand, cand_cap, depth, stage_begin, stage_end, deep, deep_cap, integ_stride,
        cand_stride);
    return cudaGetLastError();
}

cudaError_t launch_cascade_tail_tab(const PlanDev *plan, const DevCascade *meta, const DevCascade &hmeta, const TailStump *tstumps,
                                    const double *tbase, const uint32_t *sum, const uint2 *tail, int *counters, uint32_t *cand,
                                    int cand_cap, int16_t *depth, int stage_begin, int stage_end, uint2 *deep, int deep_cap,
                                    cudaStream_t st)
{
    return launch_tail_tab_t<false>(plan, meta, hmeta, tstumps, tbase, sum, tail, counters, cand, cand_cap, depth, stage_begin, stage_end,
                                    deep, deep_cap, st, 0, 0);
}

cudaError_t launch_cascade_tail_tab_batch(const PlanDev *plan, const DevCascade *meta, const DevCascade &hmeta, const TailStump *tstumps,
                                          const double *tbase, const uint32_t *sum, size_t integ_stride, const uint2 *queue, int queue_cap,
                                          int *counters, uint32_t *cand, int cand_stride, cudaStream_t st)
{
    return launch_tail_tab_t<true>(plan, meta, hmeta, tstumps, tbase, sum, queue, counters, cand, cand_stride, nullptr, 1, hmeta.nstages,
                                   nullptr, queue_cap, st, integ_stride, cand_stride);
}

cudaError_t launch_stage0_rows_gen(const PlanDev *plan, int total_rows, const DevCascade *meta, const GenModel &g,
                                   const uint32_t *sum, const uint32_t *sq, const uint32_t *tilt, float *vnf,
                                   uint32_t *bits_alive, int *counters, int16_t *depth, cudaStream_t st)
{
    k_stage0_rows_gen<<<(total_rows + 7) / 8, 256, 0, st>>>(plan, total_rows, meta, g, sum, sq, tilt, vnf, bits_alive, counters, depth);
    return cudaGetLastError();
}

cudaError_t launch_queue_stages_gen(const PlanDev *plan, const DevCascade *meta, const GenModel &g, const uint32_t *sum,
                                    const uint32_t *tilt, const uint2 *queue, int *counters, uint32_t *cand, int cand_cap,
                                    int16_t *depth, int nblocks, int order_free, cudaStream_t st)
{
    if (order_free) k_queue_stages_gen_warp<<<nblocks, 256, 0, st>>>(plan, meta, g, sum, tilt, queue, counters, cand, cand_cap, depth, 1, 0);
    else k_queue_stages_gen<<<nblocks, 256, 0, st>>>(plan, meta, g, sum, tilt, queue, counters, cand, cand_cap, depth);
    return cudaGetLastError();
}

// Large plans: stages 1 .. nstages-1 in passes of growing depth with compaction in between (k_queue_range_gen), ping-pong
// between the two queues; the few windows that get past the scheduled ranges finish with one warp each (order-free
// models) or in one more thread-per-window pass.  counters[8 + i] counts the survivors of pass i.
cudaError_t launch_queue_stages_gen_staged(const PlanDev *plan, const DevCascade *meta, const GenModel &g, const uint32_t *sum,
                                           const uint32_t *tilt, uint2 *queue_a, uint2 *queue_b, int qcap, int *counters,
                                           uint32_t *cand, int cand_cap, int16_t *depth, int nstages, int order_free,
                                           cudaStream_t st, int *nlaunch)
{
    static const int width[] = {1, 1, 1, 2, 4};                  // stages per pass: [1,2) [2,3) [3,4) [4,6) [6,10)
    const int nblocks = 148 * 8;
    uint2 *qin = queue_a, *qout = queue_b;
    int cin = 0, sb = 1, pass = 0;
    for (; pass < 5 && sb < nstages; pass++) {
        const int se = sb + width[pass] < nstages ? sb + width[pass] : nstages;
        const int final = se == nstages;
        k_queue_range_gen<<<nblocks, 256, 0, st>>>(plan, meta, g, sum, tilt, qin, qout, qcap, counters, cin, 8 + pass, cand, cand_cap,
                                                   depth, sb, se, final);
        (*nlaunch)++;
        cin = 8 + pass; sb = se;
        uint2 *t = qin; qin = qout; qout = t;
    }
    if (sb < nstages) {
        if (order_free)
            k_queue_stages_gen_warp<<<nblocks, 256, 0, st>>>(plan, meta, g, sum, tilt, qin, counters, cand, cand_cap, depth, sb, cin);
        else
            k_queue_range_gen<<<nblocks, 256, 0, st>>>(plan, meta, g, sum, tilt, qin, qout, qcap, counters, cin, 15, cand, cand_cap, depth,
                                                       sb, nstages, 1);
        (*nlaunch)++;
    }
    return cudaGetLastError();
}

cudaError_t launch_stage0_rows_p(const Stage0Params &sp, cudaStream_t st)
{
    k_stage0_rows_p<false><<<(sp.total_rows + 7) / 8, 256, 0, st>>>(sp);
    return cudaGetLastError();
}

cudaError_t launch_stage0_rows_p_batch(const Stage0Params &sp, int n, cudaStream_t st)
{
    k_stage0_rows_p<true><<<dim3((sp.total_rows + 7) / 8, n), 256, 0, st>>>(sp);
    return cudaGetLastError();
}
