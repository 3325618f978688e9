// kernels_group.cu — K8: on-device cv::groupRectangles(minNeighbors, 0.2) + the final clip of
// CascadeClassifier::detectMultiScale (SURVEY.md A.7, A.8; call sites kmsfacedetect.cpp:809-811 etc.).
//
// cv::partition's class labels depend only on the connected components of the SimilarRects graph and on
// the order of first members, so its sequential union-find with rank is replaced by: canonical ordering of
// the candidates (rank sort on the packed window id = scale -> y -> x, OpenCV's single-thread order), a
// similarity bit-matrix built by many blocks, then min-label propagation in one block (labels in shared
// memory, one warp per matrix row, rows prefetched) — dense clusters converge in two or three sweeps, and
// every component ends up labelled by its first member.
//
// Above NV_GROUP_UF_MIN candidates (a permissive model over a full frame: haarcascade_smile.xml leaves 15 000 on a 1080p
// image) the n x n matrix is the whole cost, so the components are built another way: every candidate looks for similar
// ones only where they can be — the canonical order is (level, row, column), similar rectangles differ in size by at most
// 2 delta, i.e. sit on a few neighbouring levels, and in rows within delta — and links them with a lock-free union-find
// whose root is the smallest index (uf_link inside k_adj, many blocks).  Same components, same labels (first member), so the rest
// of k_group is shared.
//
// Scores (SCORES = true, nv_ctx_set_scores): the warp that ranks a candidate also evaluates the candidate's LAST stage —
// detectMultiScale3's levelWeights is that stage's sum — and the grouping passes on, per output rectangle, the class size
// (detectMultiScale2's numDetections) and the largest member weight.  The bulk cascade kernels keep no stage sums, so the
// stage is evaluated again here, in the reference's arithmetic whatever kernel produced the candidate: the variance
// factor as in stage 0, one lane per weak classifier, and the double sum formed in XML order by one shuffle per
// classifier, so it is exact for every cascade without the order-free certificate.
#include "cascade_eval.cuh"


#define GROUP_SMEM_LABELS NV_GROUP_UF_MIN      // the matrix path keeps its labels in shared memory

__device__ __forceinline__ bool similar_rects(const int4 &a, const int4 &b, double eps)
{
    double delta = eps * (double)(min(a.z, b.z) + min(a.w, b.w)) * 0.5;
    return (double)abs(a.x - b.x) <= delta && (double)abs(a.y - b.y) <= delta &&
           (double)abs(a.x + a.z - b.x - b.z) <= delta && (double)abs(a.y + a.w - b.y - b.w) <= delta;
}

// sum of the last stage at candidate `key`, evaluated by the whole warp (every lane returns it)
__device__ __forceinline__ double last_stage_weight(const ScoreArgs &sa, const PlanDev *__restrict__ plan, uint32_t key, int lane)
{
    const int l = key >> 26, iy = (key >> 13) & 8191, ix = key & 8191;
    const LevelDesc &L = plan->lv[l];
    LevelView v{sa.sum + L.iofs, L.ipitch, L.iplane, L.ystep};
    const size_t rowbase = (size_t)iy * L.ystep * L.ipitch;
    const uint32_t *wb = v.sum + rowbase + ix;
    float vnf = 0.f;
    if (!sa.g.subset) {                                           // Haar: the variance factor exactly as stage 0 forms it
        const int ww = plan->win_w, wh = plan->win_h;
        const int c00 = corner(v, 1, 1), c10 = corner(v, ww - 1, 1), c01 = corner(v, 1, wh - 1), c11 = corner(v, ww - 1, wh - 1);
        const uint32_t *qb = sa.sq + L.iofs + rowbase + ix;
        const double area = (double)((ww - 2) * (wh - 2));
        const int valsum = (int)(__ldg(wb + c00) - __ldg(wb + c10) - __ldg(wb + c01) + __ldg(wb + c11));
        const uint32_t valsq = __ldg(qb + c00) - __ldg(qb + c10) - __ldg(qb + c01) + __ldg(qb + c11);
        const double nf = __dsub_rn(__dmul_rn(area, (double)valsq), __dmul_rn((double)valsum, (double)valsum));
        vnf = __double2float_rn(__ddiv_rn(1.0, __dsqrt_rn(nf)));  // nf > 0: the candidate passed the variance test
    }
    const uint32_t *tb = sa.tilt ? sa.tilt + L.iofs + rowbase + ix * L.ystep : nullptr;
    const int st = sa.meta->nstages - 1, t0 = sa.meta->stage_first[st], t1 = sa.meta->stage_first[st + 1];
    double w = 0.;
    for (int t = t0; t < t1; t += 32) {
        const int k = t + lane;
        double leaf = 0.;
        if (k < t1)
            leaf = sa.general ? gen_stage_sum(sa.g, k, k + 1, wb, v, tb, L.ipitch, vnf)
                              : (double)stump_leaf(wb, v, load_stump(sa.stumps + k), vnf);
        const int m = min(32, t1 - t);
        for (int j = 0; j < m; j++) w = __dadd_rn(w, __shfl_sync(0xffffffffu, leaf, j));     // XML order
    }
    return w;
}

// order-preserving map of a double onto uint64 (atomicMax over class members) and back
__device__ __forceinline__ unsigned long long weight_key(double w)
{
    const unsigned long long u = (unsigned long long)__double_as_longlong(w);
    return (u >> 63) ? ~u : u | 0x8000000000000000ull;
}
__device__ __forceinline__ double weight_of_key(unsigned long long k)
{
    return __longlong_as_double((long long)((k >> 63) ? k & 0x7fffffffffffffffull : ~k));
}

// rank sort + candidate rectangles (A.6: cvRound of FLOAT products)
template <bool SCORES>
__device__ __forceinline__ void cand_sort_body(const PlanDev *__restrict__ plan, int n, const uint32_t *__restrict__ cand,
                                               uint32_t *sorted, int4 *rects, int *label, const ScoreArgs &sa)
{
    // one WARP per candidate: its rank is counted 32 keys at a time and summed by a warp reduction (a thread per candidate
    // walked all n keys alone — n threads busy, each for n dependent iterations)
    const int lane = threadIdx.x & 31, nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += nwarps) {
        const uint32_t key = __ldg(cand + i);
        int rank = 0;
        for (int j = lane; j < n; j += 32) rank += __ldg(cand + j) < key;
        rank = __reduce_add_sync(0xffffffffu, rank);
        double wt = 0.;
        if (SCORES) wt = last_stage_weight(sa, plan, key, lane);
        if (lane) continue;
        int l = key >> 26, iy = (key >> 13) & 8191, ix = key & 8191;
        const LevelDesc &L = plan->lv[l];
        float sc = L.scale;
        int4 r;
        r.x = __float2int_rn(__fmul_rn(__int2float_rn(ix * L.ystep), sc));
        r.y = __float2int_rn(__fmul_rn(__int2float_rn(iy * L.ystep), sc));
        r.z = __float2int_rn(__fmul_rn(__int2float_rn(plan->win_w), sc));
        r.w = __float2int_rn(__fmul_rn(__int2float_rn(plan->win_h), sc));
        sorted[rank] = key;
        rects[rank] = r;
        if (SCORES) sa.w[rank] = wt;
        if (label) label[rank] = rank;                            // union-find forest of the large-n path
    }
}

template <bool SCORES>
__global__ void __launch_bounds__(256)
k_cand_sort(const PlanDev *__restrict__ plan, const int *__restrict__ counters, const uint32_t *__restrict__ cand,
            int cand_cap, uint32_t *__restrict__ sorted, int4 *__restrict__ rects, int *__restrict__ label, const ScoreArgs sa)
{
    cand_sort_body<SCORES>(plan, min(counters[1], cand_cap), cand, sorted, rects, label, sa);
}

__device__ __forceinline__ int uf_find(int *L, int a)
{
    int p;
    while ((p = ((volatile int *)L)[a]) != a) a = p;
    return a;
}
__device__ __forceinline__ void uf_union(int *L, int a, int b)
{
    bool done;
    do {
        a = uf_find(L, a);
        b = uf_find(L, b);
        if (a < b) { int old = atomicMin(&L[b], a); done = old == b; b = old; }
        else if (b < a) { int old = atomicMin(&L[a], b); done = old == a; a = old; }
        else done = true;
    } while (!done);
}
__device__ __forceinline__ int key_lower_bound(const uint32_t *keys, int n, uint32_t key)
{
    int lo = 0, hi = n;
    while (lo < hi) { int mid = (lo + hi) >> 1; if (keys[mid] < key) lo = mid + 1; else hi = mid; }
    return lo;
}

// large n: candidate i against the candidates AFTER it in canonical order that can be similar to it
__device__ void uf_link(const PlanDev *__restrict__ plan, int n, const uint32_t *sorted, const int4 *rects, int *label, double eps)
{
    const int nlevels = plan->nlevels;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t key = sorted[i];
        const int l = key >> 26;
        const int4 a = rects[i];
        for (int l2 = l; l2 < nlevels; l2++) {
            const LevelDesc &L2 = plan->lv[l2];
            const int w2 = __float2int_rn(__fmul_rn(__int2float_rn(plan->win_w), L2.scale));
            const int h2 = __float2int_rn(__fmul_rn(__int2float_rn(plan->win_h), L2.scale));
            // sizes grow with the level: delta is set by level l, and |w1 - w2| <= 2 delta is necessary for similarity
            const double delta = eps * (double)(min(a.z, w2) + min(a.w, h2)) * 0.5;
            if ((double)abs(w2 - a.z) > 2.0 * delta || (double)abs(h2 - a.w) > 2.0 * delta) break;
            const double step = (double)L2.ystep * (double)L2.scale;
            int lo = (int)floor(((double)a.y - delta - 1.0) / step) - 1, hi = (int)ceil(((double)a.y + delta + 1.0) / step) + 1;
            lo = max(lo, 0); hi = min(hi, 8190);
            int j0 = key_lower_bound(sorted, n, ((uint32_t)l2 << 26) | ((uint32_t)lo << 13));
            const int j1 = key_lower_bound(sorted, n, ((uint32_t)l2 << 26) | ((uint32_t)(hi + 1) << 13));
            if (l2 == l) j0 = max(j0, i + 1);
            for (int j = j0; j < j1; j++)
                if (similar_rects(a, rects[j], eps)) uf_union(label, i, j);
        }
    }
}

// similarity bit-matrix: word (i, w) holds the similarity of candidate i with candidates 32w .. 32w+31
__device__ __forceinline__ void adj_body(const PlanDev *__restrict__ plan, int n, const uint32_t *sorted, const int4 *rects,
                                         uint32_t *adj, int *label, double eps)
{
    const int nw = (n + 31) >> 5;
    if (n > NV_GROUP_UF_MIN) { uf_link(plan, n, sorted, rects, label, eps); return; }     // large n: components by union-find
    // one WARP per matrix word, one pair per lane, the word assembled by a vote (a thread per word tested its 32 pairs one
    // after the other: a chain of 32 dependent iterations where this is one)
    const int lane = threadIdx.x & 31, nwarps = (gridDim.x * blockDim.x) >> 5;
    const int total = n * nw;                                     // n <= NV_GROUP_UF_MIN: fits an int
    for (int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; t < total; t += nwarps) {
        const int i = t / nw, w = t - i * nw, j = w * 32 + lane;
        const int4 a = rects[i];
        const bool bit = j < n && j != i && similar_rects(a, rects[min(j, n - 1)], eps);
        const uint32_t m = __ballot_sync(0xffffffffu, bit);
        if (lane == 0) adj[t] = m;
    }
}

__global__ void __launch_bounds__(256)
k_adj(const PlanDev *__restrict__ plan, const int *__restrict__ counters, int cand_cap, const uint32_t *__restrict__ sorted,
      const int4 *__restrict__ rects, uint32_t *__restrict__ adj, int *__restrict__ label, double eps)
{
    adj_body(plan, min(counters[1], cand_cap), sorted, rects, adj, label, eps);
}

#ifndef NV_GROUP_THREADS
#define NV_GROUP_THREADS 1024
#endif
#define NV_GROUP_WARPS (NV_GROUP_THREADS / 32)
// exclusive rank of a 0/1 flag across the block, with a running carry
template <int NT>
__device__ __forceinline__ int block_flag_rank(bool flag, int &carry, int *s_warp)
{
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t m = __ballot_sync(0xffffffffu, flag);
    if (lane == 0) s_warp[warp] = __popc(m);
    __syncthreads();
    int before = 0, total = 0;
    for (int k = 0; k < (NT / 32); k++) { int c = s_warp[k]; if (k < warp) before += c; total += c; }
    int pos = carry + before + __popc(m & ((1u << lane) - 1u));
    carry += total;
    __syncthreads();
    return pos;
}

// grp scratch layout (ints): label[cap] | cls[cap] | acc[5*cap] (x,y,w,h,count) | keep[cap]
// SCORES: output i also gets its neighbour count and level weight, in the result block after the rectangles
template <int NT, bool SCORES>
__device__ __forceinline__ void group_body(int *counters, int cand_cap, const int4 *rects, const uint32_t *adj, int *grp,
                                           int min_neighbors, double eps, int img_w, int img_h, uint8_t *result, int result_cap,
                                           uint8_t *host_result, const ScoreArgs &sa)
{
    __shared__ int s_warp[32];
    int tid = threadIdx.x;
    int n = min(counters[1], cand_cap), nw = (n + 31) >> 5;
    ResultHeader *hdr = reinterpret_cast<ResultHeader *>(result);
    int4 *out = reinterpret_cast<int4 *>(result + sizeof(ResultHeader));
    // host_result: the context's page-locked result block, mapped into the device's address space.  Header and the first
    // NV_RESULT_INLINE rectangles are written there as well, straight over PCIe, so that no device-to-host copy follows
    // the launch (one node less in every call's graph).
    int4 *hout = host_result ? reinterpret_cast<int4 *>(host_result + sizeof(ResultHeader)) : nullptr;
    double *out_w = reinterpret_cast<double *>(out + result_cap), *hout_w = hout ? reinterpret_cast<double *>(hout + result_cap) : nullptr;
    int *out_n = reinterpret_cast<int *>(out_w + result_cap), *hout_n = hout ? reinterpret_cast<int *>(hout_w + result_cap) : nullptr;
    auto put_scores = [&](int pos, int nb, double w) {
        out_w[pos] = w; out_n[pos] = nb;
        if (hout && pos < NV_RESULT_INLINE) { hout_w[pos] = w; hout_n[pos] = nb; }
    };
    extern __shared__ int s_label[];                 // min(n, GROUP_SMEM_LABELS) labels; global scratch beyond that
    __shared__ int s_changed;
    const bool uf = n > NV_GROUP_UF_MIN;                          // labels already final in grp (uf_link in k_adj, flattened below)
    volatile int *label = uf ? grp : s_label;
    int *cls = grp + cand_cap, *acc = grp + 2 * cand_cap, *keep = grp + 7 * cand_cap;
    int nout = 0;

    if (min_neighbors <= 0) {
        // no grouping: canonical-order candidates, clipped; empty intersections are dropped (A.8)
        int carry = 0;
        for (int i0 = 0; i0 < n; i0 += NT) {
            int i = i0 + tid;
            int4 r = make_int4(0, 0, 0, 0);
            bool k = false;
            if (i < n) {
                r = rects[i];
                int x0 = max(r.x, 0), y0 = max(r.y, 0), x1 = min(r.x + r.z, img_w), y1 = min(r.y + r.w, img_h);
                k = x1 > x0 && y1 > y0;
                r = make_int4(x0, y0, x1 - x0, y1 - y0);
            }
            int pos = block_flag_rank<NT>(k, carry, s_warp);
            if (k && pos < result_cap) {
                out[pos] = r; if (hout && pos < NV_RESULT_INLINE) hout[pos] = r;
                if (SCORES) put_scores(pos, 1, sa.w[i]);
            }
        }
        nout = carry;
    } else {
        if (!uf) for (int i = tid; i < n; i += NT) label[i] = i;
        else {                                                    // flatten the forest k_adj linked: roots stay put, paths only get shorter
            for (int i = tid; i < n; i += NT) { const int r = uf_find(grp, i); if (r != i) grp[i] = r; }
        }
        __syncthreads();
        // min-label propagation until a fixed point: one warp per candidate row.  A lane fetches one adjacency word of the row
        // (the next row's while the current one is reduced); the non-zero words are then taken one at a time by the WHOLE warp,
        // one bit per lane — in the clusters of a frame with faces a word holds 20-30 set bits, and walking them with a lane per
        // word (the first version) left 25 lanes idle behind seven that looped: 59 % of the kernel's instructions on config 3.
        const int lane = tid & 31, warp = tid >> 5;
        for (; !uf;) {
            if (tid == 0) s_changed = 0;
            __syncthreads();
            uint32_t nxt = (warp < n && lane < nw) ? adj[(size_t)warp * nw + lane] : 0u;
            for (int i = warp; i < n; i += (NT / 32)) {
                int m = 0x7fffffff;
                uint32_t b = nxt;
                if (i + (NT / 32) < n) nxt = lane < nw ? adj[(size_t)(i + (NT / 32)) * nw + lane] : 0u;
                for (int w0 = 0; w0 < nw; w0 += 32) {
                    if (w0 > 0) b = w0 + lane < nw ? adj[(size_t)i * nw + w0 + lane] : 0u;      // more than 1024 candidates
                    uint32_t nz = __ballot_sync(0xffffffffu, b != 0u);
                    while (nz) {
                        const int src = __ffs(nz) - 1;
                        nz &= nz - 1;
                        const uint32_t bw = __shfl_sync(0xffffffffu, b, src);
                        if ((bw >> lane) & 1u) m = min(m, label[(w0 + src) * 32 + lane]);
                    }
                }
                m = __reduce_min_sync(0xffffffffu, m);
                if (lane == 0) {
                    int c = label[i];
                    m = min(m, c);
                    m = min(m, label[m]);
                    if (m < c) { label[i] = m; s_changed = 1; }
                }
            }
            __syncthreads();
            int ch = s_changed;
            __syncthreads();
            if (!ch) break;
        }
        // classes numbered by their first member (= the component's minimum index)
        int carry = 0;
        for (int i0 = 0; i0 < n; i0 += NT) {
            int i = i0 + tid;
            bool root = i < n && label[i] == i;
            int pos = block_flag_rank<NT>(root, carry, s_warp);
            if (root) cls[i] = pos;
        }
        int ncls = carry;
        for (int i = tid; i < 5 * ncls; i += NT) acc[i] = 0;
        if (SCORES) for (int c = tid; c < ncls; c += NT) sa.cls_wmax[c] = 0ull;     // below the key of any finite weight
        __syncthreads();
        for (int i = tid; i < n; i += NT) {
            int c = cls[label[i]];
            int4 r = rects[i];
            atomicAdd(&acc[5 * c + 0], r.x); atomicAdd(&acc[5 * c + 1], r.y);
            atomicAdd(&acc[5 * c + 2], r.z); atomicAdd(&acc[5 * c + 3], r.w);
            atomicAdd(&acc[5 * c + 4], 1);
            if (SCORES) atomicMax(&sa.cls_wmax[c], weight_key(sa.w[i]));
        }
        __syncthreads();
        for (int c = tid; c < ncls; c += NT) {
            float s = __fdiv_rn(1.f, __int2float_rn(acc[5 * c + 4]));
            for (int k = 0; k < 4; k++) acc[5 * c + k] = __float2int_rn(__fmul_rn(__int2float_rn(acc[5 * c + k]), s));
        }
        __syncthreads();
        // classes with enough members, in class order (the containment test only ever looks at those)
        int nk = 0;
        for (int i0 = 0; i0 < ncls; i0 += NT) {
            int i = i0 + tid;
            bool k = i < ncls && acc[5 * i + 4] > min_neighbors;
            int pos = block_flag_rank<NT>(k, nk, s_warp);
            if (k) keep[pos] = i;
        }
        __syncthreads();
        // drop a class that lies inside a clearly stronger one (A.7)
        int *alive = cls;                                   // cls[] is no longer needed: reuse as the survivor flags
        __syncthreads();
        for (int a = tid; a < nk; a += NT) {
            int i = keep[a];
            int n1 = acc[5 * i + 4], x1 = acc[5 * i], y1 = acc[5 * i + 1], w1 = acc[5 * i + 2], h1 = acc[5 * i + 3];
            bool k = true;
            for (int b = 0; b < nk && k; b++) {
                int j = keep[b];
                if (j == i) continue;
                int n2 = acc[5 * j + 4];
                int x2 = acc[5 * j], y2 = acc[5 * j + 1], w2 = acc[5 * j + 2], h2 = acc[5 * j + 3];
                int dx = __double2int_rn(__dmul_rn((double)w2, eps)), dy = __double2int_rn(__dmul_rn((double)h2, eps));
                if (x1 >= x2 - dx && y1 >= y2 - dy && x1 + w1 <= x2 + w2 + dx && y1 + h1 <= y2 + h2 + dy &&
                    (n2 > max(3, n1) || n1 < 3)) k = false;
            }
            alive[a] = k;
        }
        __syncthreads();
        carry = 0;
        for (int a0 = 0; a0 < nk; a0 += NT) {
            int a = a0 + tid;
            bool k = false;
            int4 r = make_int4(0, 0, 0, 0);
            if (a < nk && alive[a]) {
                int i = keep[a];
                int x0 = max(acc[5 * i], 0), y0 = max(acc[5 * i + 1], 0);
                int x1 = min(acc[5 * i] + acc[5 * i + 2], img_w), y1 = min(acc[5 * i + 1] + acc[5 * i + 3], img_h);
                k = x1 > x0 && y1 > y0;
                r = make_int4(x0, y0, x1 - x0, y1 - y0);
            }
            int pos = block_flag_rank<NT>(k, carry, s_warp);
            if (k && pos < result_cap) {
                out[pos] = r; if (hout && pos < NV_RESULT_INLINE) hout[pos] = r;
                if (SCORES) { const int i = keep[a]; put_scores(pos, acc[5 * i + 4], weight_of_key(sa.cls_wmax[i])); }
            }
        }
        nout = carry;
    }
    __syncthreads();                                     // every thread has read its counters
    if (tid == 0) {
        hdr->n_out = min(nout, result_cap);
        hdr->n_cand = counters[1];
        hdr->n_alive = counters[0];
        hdr->overflow = counters[2] | (nout > result_cap) | (counters[1] > cand_cap);
        if (host_result) *reinterpret_cast<ResultHeader *>(host_result) = *hdr;
        for (int i = 0; i < 16; i++) counters[i] = 0;    // the call's last kernel leaves the counters ready for the next call
    }
}

template <bool SCORES>
__global__ void __launch_bounds__(NV_GROUP_THREADS)
k_group(int *__restrict__ counters, int cand_cap, const int4 *__restrict__ rects, const uint32_t *__restrict__ adj,
        int *__restrict__ grp, int min_neighbors, double eps, int img_w, int img_h, uint8_t *__restrict__ result,
        int result_cap, uint8_t *__restrict__ host_result, const ScoreArgs sa)
{
    group_body<NV_GROUP_THREADS, SCORES>(counters, cand_cap, rects, adj, grp, min_neighbors, eps, img_w, img_h, result, result_cap,
                                         host_result, sa);
}

// Small plans (a config-1 frame, a nested ROI: a few dozen candidates): canonical order, similarity matrix and grouping by
// ONE block in one launch — three launches of a few microseconds each were a sixth of such a call.  The arrays pass
// between the phases through global memory behind block barriers, so none of them is a read-only (__restrict__ const)
// parameter here.  256 threads: with the few dozen candidates of such a call 24 of a 1024-thread block's warps only run loop
// control and barriers.  (Keeping keys, rectangles, matrix and class tables of up to 256 candidates in shared memory was
// measured too: no change, 19 us under ncu either way — the launch is a chain of short dependent phases of one block.)
//
// BATCH: one block per image of a batch, image blockIdx.y (gridDim.x stays 1, so the bodies' grid-stride loops cover the
// image's own candidates).  The image's counters are counters + 16 * (1 + image), its candidates the segment at
// image * cand_stride, its scratch and result block at image times their sizes; block 0 also clears the batch's shared
// counter block (counters[0 .. 15]: queue count and ticket).
#define NV_GROUP_FUSED_THREADS 256
template <bool SCORES, bool BATCH>
__global__ void __launch_bounds__(NV_GROUP_FUSED_THREADS)
k_group_fused(const PlanDev *__restrict__ plan, int *counters, const uint32_t *__restrict__ cand, int cand_cap, uint32_t *sorted,
              int4 *rects, uint32_t *adj, int *grp, int min_neighbors, double eps, int img_w, int img_h, uint8_t *result,
              int result_cap, uint8_t *host_result, const ScoreArgs sa, int cand_stride = 0, size_t adj_stride = 0,
              size_t result_stride = 0)
{
    if (BATCH) {
        const int img = blockIdx.y;
        if (img == 0 && threadIdx.x < 16) counters[threadIdx.x] = 0;
        counters += 16 * (1 + img);
        cand += img * (size_t)cand_stride;
        sorted += img * (size_t)cand_cap; rects += img * (size_t)cand_cap; grp += img * 8 * (size_t)cand_cap; adj += img * adj_stride;
        result += img * result_stride; host_result += img * result_stride;
    }
    const int n = min(counters[1], cand_cap);
    cand_sort_body<SCORES>(plan, n, cand, sorted, rects, min_neighbors > 0 ? grp : nullptr, sa);
    __syncthreads();
    if (min_neighbors > 0) {
        adj_body(plan, n, sorted, rects, adj, grp, eps);
        __syncthreads();
    }
    group_body<NV_GROUP_FUSED_THREADS, SCORES>(counters, cand_cap, rects, adj, grp, min_neighbors, eps, img_w, img_h, result, result_cap,
                                               host_result, sa);
}

template <bool SCORES>
static cudaError_t launch_group_t(const PlanDev *plan, int *counters, const uint32_t *cand, int cand_cap, uint32_t *cand_sorted,
                                  int4 *cand_rects, uint32_t *adj, int *grp, int min_neighbors, double eps, int img_w, int img_h,
                                  uint8_t *result, int result_cap, int nblocks, cudaStream_t st, int *nlaunch, bool fused,
                                  uint8_t *host_result, const ScoreArgs &sa)
{
    if (fused) {
        k_group_fused<SCORES, false><<<1, NV_GROUP_FUSED_THREADS, GROUP_SMEM_LABELS * sizeof(int), st>>>(
            plan, counters, cand, cand_cap, cand_sorted, cand_rects, adj, grp, min_neighbors, eps, img_w, img_h, result, result_cap,
            host_result, sa);
        (*nlaunch)++;
        return cudaGetLastError();
    }
    k_cand_sort<SCORES><<<nblocks, 256, 0, st>>>(plan, counters, cand, cand_cap, cand_sorted, cand_rects, min_neighbors > 0 ? grp : nullptr,
                                                 sa);
    (*nlaunch)++;
    if (min_neighbors > 0) {
        k_adj<<<nblocks, 256, 0, st>>>(plan, counters, cand_cap, cand_sorted, cand_rects, adj, grp, eps);
        (*nlaunch)++;
    }
    k_group<SCORES><<<1, NV_GROUP_THREADS, GROUP_SMEM_LABELS * sizeof(int), st>>>(counters, cand_cap, cand_rects, adj, grp, min_neighbors,
                                                                                  eps, img_w, img_h, result, result_cap, host_result, sa);
    (*nlaunch)++;
    return cudaGetLastError();
}

cudaError_t launch_group(const PlanDev *plan, int *counters, const uint32_t *cand, int cand_cap, uint32_t *cand_sorted,
                         int4 *cand_rects, uint32_t *adj, int *grp, int min_neighbors, double eps, int img_w, int img_h,
                         uint8_t *result, int result_cap, int nblocks, cudaStream_t st, int *nlaunch, bool fused, uint8_t *host_result,
                         const ScoreArgs *scores)
{
    if (scores)
        return launch_group_t<true>(plan, counters, cand, cand_cap, cand_sorted, cand_rects, adj, grp, min_neighbors, eps, img_w, img_h,
                                    result, result_cap, nblocks, st, nlaunch, fused, host_result, *scores);
    return launch_group_t<false>(plan, counters, cand, cand_cap, cand_sorted, cand_rects, adj, grp, min_neighbors, eps, img_w, img_h,
                                 result, result_cap, nblocks, st, nlaunch, fused, host_result, ScoreArgs{});
}

cudaError_t launch_group_batch(const PlanDev *plan, int n, int *counters, const uint32_t *cand, int cand_stride, int cap, uint32_t *cand_sorted,
                               int4 *cand_rects, uint32_t *adj, size_t adj_stride, int *grp, int min_neighbors, double eps, int img_w,
                               int img_h, uint8_t *result, uint8_t *host_result, size_t result_stride, cudaStream_t st)
{
    k_group_fused<false, true><<<dim3(1, n), NV_GROUP_FUSED_THREADS, GROUP_SMEM_LABELS * sizeof(int), st>>>(
        plan, counters, cand, cap, cand_sorted, cand_rects, adj, grp, min_neighbors, eps, img_w, img_h, result, cap, host_result,
        ScoreArgs{}, cand_stride, adj_stride, result_stride);
    return cudaGetLastError();
}
