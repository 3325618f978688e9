// context.cu — the C ABI of libnubovca.so (include/nubovca.h): cascade objects, per-element contexts, the
// per-frame plan (scale list, level geometry, coefficient tables), and the stream-ordered pipelines that
// replace the OpenCV call blocks of the reference elements.  No host decision is taken between the H2D copy
// of a frame and the D2H copy of its rectangles: candidate counts stay on the device.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>

#include "internal.h"

#define NV_VERSION_STR "nubovca-b200 0.1 (sm_100a)"
#define CAND_CAP 8192              // initial raw-candidate capacity; grows on demand (collect() re-runs the call)
#define CAND_CAP_GROUPED 65536     // hard limit of a grouped call (rank sort and union-find scratch grow with it; allocated on demand only)
#define CAND_CAP_RAW 131072

extern "C" const char *nv_version(void) { return NV_VERSION_STR; }

extern "C" int nv_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

// ------------------------------------------------------------------------------------------------
// cascade
// ------------------------------------------------------------------------------------------------
extern "C" int nv_cascade_load(const char *xml_path, nv_cascade **out)
{
    if (!xml_path || !out) { nv_set_error("nv_cascade_load: null argument"); return NV_ERR_ARG; }
    *out = nullptr;
    static std::atomic<unsigned long long> next_uid{1};
    nv_cascade *c = new nv_cascade();
    c->uid = next_uid.fetch_add(1);
    int rc = nv_parse_cascade_xml(xml_path, &c->h);
    if (rc != NV_OK) { delete c; return rc; }
    const HostCascade &h = c->h;
    memset(&c->meta, 0, sizeof c->meta);
    c->meta.win_w = h.win_w; c->meta.win_h = h.win_h;
    c->meta.nstages = (int)h.stage_ntrees.size(); c->meta.nstumps = (int)h.stump_feat.size();
    int acc = 0;
    for (int s = 0; s < c->meta.nstages; s++) {
        c->meta.stage_first[s] = acc;
        acc += h.stage_ntrees[s];
        c->meta.stage_thr[s] = h.stage_thr[s] - 1e-5f;            // THRESHOLD_EPS, float arithmetic
    }
    c->meta.stage_first[c->meta.nstages] = acc;
    c->stumps.resize(h.stump_feat.size());
    for (size_t i = 0; i < h.stump_feat.size(); i++) {
        DevStump &d = c->stumps[i];
        memset(&d, 0, sizeof d);
        const int *r = &h.feat_rect[(size_t)h.stump_feat[i] * 12];
        const float *w = &h.feat_weight[(size_t)h.stump_feat[i] * 3];
        for (int k = 0; k < 3; k++) {
            d.r[k] = (uint32_t)r[4 * k] | ((uint32_t)r[4 * k + 1] << 8) | ((uint32_t)r[4 * k + 2] << 16) |
                     ((uint32_t)r[4 * k + 3] << 24);
            d.w[k] = w[k];
        }
        d.thr = h.stump_thr[i]; d.left = h.stump_left[i]; d.right = h.stump_right[i];
    }
    build_tail_stumps(c);
    *out = c;
    return NV_OK;
}

extern "C" int nv_cascade_get_info(const nv_cascade *c, nv_cascade_info *info)
{
    if (!c || !info) { nv_set_error("nv_cascade_get_info: null argument"); return NV_ERR_ARG; }
    info->win_w = c->h.win_w; info->win_h = c->h.win_h;
    info->nstages = (int)c->h.stage_ntrees.size(); info->nstumps = (int)c->h.stump_feat.size();
    info->nfeatures = (int)c->h.feat_weight.size() / 3; info->n3rect = c->h.n3rect;
    info->order_free_sums = c->h.order_free;
    info->general = c->h.general; info->has_tilted = c->h.has_tilted; info->nnodes = (int)c->h.node_feat.size();
    info->lbp = c->h.lbp;
    return NV_OK;
}

extern "C" int nv_debug_cascade_stage(const nv_cascade *c, int stage, int *ntrees, float *threshold_used)
{
    if (!c || stage < 0 || stage >= c->meta.nstages) { nv_set_error("bad argument"); return NV_ERR_ARG; }
    if (ntrees) *ntrees = c->meta.stage_first[stage + 1] - c->meta.stage_first[stage];
    if (threshold_used) *threshold_used = c->meta.stage_thr[stage];
    return NV_OK;
}

extern "C" int nv_debug_cascade_stump(const nv_cascade *c, int stump, int rects12[12], float weights3[3],
                                      float thr_left_right[3])
{
    if (!c || stump < 0 || stump >= c->meta.nstumps || !rects12 || !weights3 || !thr_left_right) {
        nv_set_error("bad argument");
        return NV_ERR_ARG;
    }
    const DevStump &d = c->stumps[stump];
    for (int k = 0; k < 3; k++) {
        rects12[4 * k] = d.r[k] & 255; rects12[4 * k + 1] = (d.r[k] >> 8) & 255;
        rects12[4 * k + 2] = (d.r[k] >> 16) & 255; rects12[4 * k + 3] = d.r[k] >> 24;
        weights3[k] = d.w[k];
    }
    thr_left_right[0] = d.thr; thr_left_right[1] = d.left; thr_left_right[2] = d.right;
    return NV_OK;
}

extern "C" int nv_debug_cascade_tree(const nv_cascade *c, int tree, int cap_nodes, int *nnodes, int *feat_left_right,
                                     float *node_thr, float *leaves)
{
    if (!c || tree < 0 || tree >= (int)c->h.tree_nnodes.size() || !nnodes) { nv_set_error("bad argument"); return NV_ERR_ARG; }
    int n0 = 0, l0 = 0;
    for (int t = 0; t < tree; t++) { n0 += c->h.tree_nnodes[t]; l0 += c->h.tree_nnodes[t] + 1; }
    int nn = c->h.tree_nnodes[tree];
    *nnodes = nn;
    if (nn > cap_nodes) { nv_set_error("tree has %d nodes", nn); return NV_ERR_CAPACITY; }
    for (int i = 0; i < nn; i++) {
        if (feat_left_right) {
            feat_left_right[3 * i] = c->h.node_feat[n0 + i]; feat_left_right[3 * i + 1] = c->h.node_left[n0 + i];
            feat_left_right[3 * i + 2] = c->h.node_right[n0 + i];
        }
        if (node_thr) node_thr[i] = c->h.node_thr[n0 + i];
    }
    if (leaves) for (int i = 0; i <= nn; i++) leaves[i] = c->h.leaves[l0 + i];
    return NV_OK;
}

extern "C" int nv_debug_cascade_feature(const nv_cascade *c, int feature, int rects12[12], float weights3[3], int *tilted)
{
    if (!c || feature < 0 || feature >= (int)c->h.feat_tilted.size() || !rects12 || !weights3) { nv_set_error("bad argument"); return NV_ERR_ARG; }
    for (int i = 0; i < 12; i++) rects12[i] = c->h.feat_rect[(size_t)feature * 12 + i];
    for (int i = 0; i < 3; i++) weights3[i] = c->h.feat_weight[(size_t)feature * 3 + i];
    if (tilted) *tilted = c->h.feat_tilted[feature];
    return NV_OK;
}

extern "C" int nv_debug_cascade_subset(const nv_cascade *c, int node, int subset8[8])
{
    if (!c || !subset8 || !c->h.lbp || node < 0 || (size_t)node * 8 + 8 > c->h.node_subset.size()) { nv_set_error("bad argument"); return NV_ERR_ARG; }
    for (int k = 0; k < 8; k++) subset8[k] = c->h.node_subset[(size_t)node * 8 + k];
    return NV_OK;
}

extern "C" void nv_cascade_free(nv_cascade *c)
{
    if (!c) return;
    for (auto &kv : c->d_stumps) { cudaSetDevice(kv.first); cudaFree(kv.second); }
    for (auto &kv : c->d_meta) { cudaSetDevice(kv.first); cudaFree(kv.second); }
    for (auto &kv : c->d_tail) { cudaSetDevice(kv.first); cudaFree(kv.second); }
    for (auto &kv : c->d_tail_base) { cudaSetDevice(kv.first); cudaFree(kv.second); }
    for (auto &kv : c->d_gen) {
        cudaSetDevice(kv.first);
        cudaFree((void *)kv.second.tree); cudaFree((void *)kv.second.node); cudaFree((void *)kv.second.leaf); cudaFree((void *)kv.second.feat);
        cudaFree((void *)kv.second.subset);
    }
    delete c;
}

// Uploads a cascade's tables to `gpu` once.  Every table is built into locals and published in the maps only after
// all uploads succeeded; a failure frees what was allocated, so a later call retries from a clean state.
static int cascade_on_device(nv_cascade *c, int gpu, cudaStream_t st, const DevStump **stumps, const DevCascade **meta)
{
    std::lock_guard<std::mutex> lk(c->mu);
    (void)st;
    if (c->d_stumps.find(gpu) == c->d_stumps.end()) {
        std::vector<void *> owned;
        struct Guard {
            std::vector<void *> &v; bool keep = false;
            ~Guard() { if (!keep) for (void *p : v) cudaFree(p); }
        } guard{owned};
        auto upload = [&](const void *src, size_t bytes, void **out) -> int {
            void *d = nullptr;
            NV_CUDA(cudaMalloc(&d, bytes ? bytes : 1));
            owned.push_back(d);
            if (bytes) NV_CUDA(cudaMemcpy(d, src, bytes, cudaMemcpyHostToDevice));
            *out = d;
            return NV_OK;
        };
        int rc;
        void *ds = nullptr, *dm = nullptr, *dtree = nullptr, *dnode = nullptr, *dleaf = nullptr, *dfeat = nullptr, *dt = nullptr, *db = nullptr, *dsub = nullptr;
        if ((rc = upload(c->stumps.data(), c->stumps.size() * sizeof(DevStump), &ds)) != NV_OK) return rc;
        if ((rc = upload(&c->meta, sizeof(DevCascade), &dm)) != NV_OK) return rc;
        if (c->h.general) {
            const HostCascade &h = c->h;
            std::vector<int2> trees(h.tree_nnodes.size());
            std::vector<int4> nodes(h.node_feat.size());
            std::vector<GenFeat> feats(h.feat_tilted.size());
            int n0 = 0, l0 = 0;
            for (size_t t = 0; t < trees.size(); t++) { trees[t] = make_int2(n0, l0); n0 += h.tree_nnodes[t]; l0 += h.tree_nnodes[t] + 1; }
            for (size_t i = 0; i < nodes.size(); i++) {
                int tb; memcpy(&tb, &h.node_thr[i], 4);
                nodes[i] = make_int4(h.node_feat[i], tb, h.node_left[i], h.node_right[i]);
            }
            for (size_t f = 0; f < feats.size(); f++) {
                GenFeat &g = feats[f];
                memset(&g, 0, sizeof g);
                for (int k = 0; k < 3; k++) {
                    const int *r = &h.feat_rect[f * 12 + 4 * k];
                    g.r[k] = (uint32_t)r[0] | ((uint32_t)r[1] << 8) | ((uint32_t)r[2] << 16) | ((uint32_t)r[3] << 24);
                    g.w[k] = h.feat_weight[f * 3 + k];
                }
                g.tilted = h.feat_tilted[f];
            }
            if ((rc = upload(trees.data(), trees.size() * sizeof(int2), &dtree)) != NV_OK) return rc;
            if ((rc = upload(nodes.data(), nodes.size() * sizeof(int4), &dnode)) != NV_OK) return rc;
            if ((rc = upload(h.leaves.data(), h.leaves.size() * sizeof(float), &dleaf)) != NV_OK) return rc;
            if ((rc = upload(feats.data(), feats.size() * sizeof(GenFeat), &dfeat)) != NV_OK) return rc;
            if (h.lbp && (rc = upload(h.node_subset.data(), h.node_subset.size() * sizeof(int), &dsub)) != NV_OK) return rc;
        }
        if (c->tail_fast) {
            if ((rc = upload(c->tail_stumps.data(), c->tail_stumps.size() * sizeof(TailStump), &dt)) != NV_OK) return rc;
            if ((rc = upload(c->tail_base.data(), c->tail_base.size() * sizeof(double), &db)) != NV_OK) return rc;
        }
        guard.keep = true;                                          // everything is on the device: publish
        if (c->h.general) c->d_gen[gpu] = GenModel{(int2 *)dtree, (int4 *)dnode, (float *)dleaf, (GenFeat *)dfeat, (uint32_t *)dsub};
        if (c->tail_fast) { c->d_tail[gpu] = (TailStump *)dt; c->d_tail_base[gpu] = (double *)db; }
        c->d_meta[gpu] = (DevCascade *)dm;
        c->d_stumps[gpu] = (DevStump *)ds;
    }
    *stumps = c->d_stumps[gpu]; *meta = c->d_meta[gpu];
    return NV_OK;
}

// ------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------
template <typename T>
static int ensure(T **p, size_t *cap, size_t need, bool zero = false)
{
    if (*p && *cap >= need) return NV_OK;
    if (*p) { NV_CUDA(cudaFree(*p)); *p = nullptr; }
    size_t n = need + need / 8 + 64;
    NV_CUDA(cudaMalloc(p, n * sizeof(T)));
    if (zero) NV_CUDA(cudaMemset(*p, 0, n * sizeof(T)));
    *cap = n;
    return NV_OK;
}

// candidate-side buffers: ids, sorted ids, rects, weights, similarity bit-matrix (+ group scratch), result block
static int alloc_candidates(nv_ctx *c, int cap, bool with_adj)
{
    cudaFree(c->d_cand); cudaFree(c->d_cand_sorted); cudaFree(c->d_cand_rects); cudaFree(c->d_adj); cudaFree(c->d_result);
    cudaFree(c->d_cand_w); cudaFree(c->d_cls_wmax);
    cudaFreeHost(c->h_result);
    c->d_cand = c->d_cand_sorted = nullptr; c->d_cand_rects = nullptr; c->d_adj = nullptr; c->d_result = c->h_result = nullptr;
    c->d_cand_w = nullptr; c->d_cls_wmax = nullptr;
    c->cand_cap = cap; c->result_cap = cap; c->adj_cap = 0; c->epoch++;
    NV_CUDA(cudaMalloc(&c->d_cand, (size_t)cap * sizeof(uint32_t)));
    NV_CUDA(cudaMalloc(&c->d_cand_sorted, (size_t)cap * sizeof(uint32_t)));
    NV_CUDA(cudaMalloc(&c->d_cand_rects, (size_t)cap * sizeof(int4)));
    NV_CUDA(cudaMalloc(&c->d_cand_w, (size_t)cap * sizeof(double)));
    NV_CUDA(cudaMalloc(&c->d_cls_wmax, (size_t)cap * sizeof(unsigned long long)));
    // the similarity bit-matrix only serves frames with at most NV_GROUP_UF_MIN candidates (kernels_group.cu)
    const size_t acap = std::min<size_t>((size_t)cap, NV_GROUP_UF_MIN);
    size_t adj_words = (with_adj ? acap * ((acap + 31) / 32) : 0) + 8 * (size_t)cap;
    NV_CUDA(cudaMalloc(&c->d_adj, adj_words * sizeof(uint32_t)));
    c->adj_cap = with_adj ? cap : 0;
    c->d_grp = reinterpret_cast<int *>(c->d_adj + (adj_words - 8 * (size_t)cap));
    size_t rbytes = sizeof(ResultHeader) + (size_t)c->result_cap * (sizeof(nv_rect) + sizeof(double) + sizeof(int));
    NV_CUDA(cudaMalloc(&c->d_result, rbytes));
    NV_CUDA(cudaMallocHost(&c->h_result, rbytes));
    memset(c->h_result, 0, sizeof(ResultHeader));
    return NV_OK;
}

extern "C" int nv_ctx_create(int gpu, int max_width, int max_height, nv_ctx **out)
{
    if (!out || max_width <= 0 || max_height <= 0 || max_width > 16384 || max_height > 16384) {
        nv_set_error("nv_ctx_create: bad argument");
        return NV_ERR_ARG;
    }
    *out = nullptr;
    int ndev = nv_device_count();
    if (ndev <= 0) { nv_set_error("no CUDA device visible: libnubovca has no CPU path"); return NV_ERR_NO_DEVICE; }
    if (gpu < 0 || gpu >= ndev) { nv_set_error("gpu ordinal %d out of range (0..%d)", gpu, ndev - 1); return NV_ERR_ARG; }
    NV_CUDA(cudaSetDevice(gpu));
    nv_ctx *c = new nv_ctx();
    c->gpu = gpu; c->max_w = max_width; c->max_h = max_height;
    int rc = [&]() -> int {
        NV_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        NV_CUDA(cudaEventCreateWithFlags(&c->ev_done, cudaEventDisableTiming));
        NV_CUDA(cudaStreamCreateWithFlags(&c->stream2, cudaStreamNonBlocking));
        for (int i = 0; i < 2; i++) {
            NV_CUDA(cudaEventCreateWithFlags(&c->ev_fork[i], cudaEventDisableTiming));
            NV_CUDA(cudaEventCreateWithFlags(&c->ev_join[i], cudaEventDisableTiming));
        }
        c->frame_cap = (size_t)max_width * max_height * 4 + 4096;
        NV_CUDA(cudaMallocHost(&c->h_frame, c->frame_cap));
        NV_CUDA(cudaMalloc(&c->d_frame, c->frame_cap));
        c->gray_cap = (size_t)max_width * max_height + 256;
        NV_CUDA(cudaMalloc(&c->d_gray, c->gray_cap));
        NV_CUDA(cudaMalloc(&c->d_hist, 260 * sizeof(int)));     // 256 bins + the prep kernels' last-block ticket
        NV_CUDA(cudaMemset(c->d_hist, 0, 260 * sizeof(int)));
        NV_CUDA(cudaMalloc(&c->d_lut, 512));
        uint8_t ident[256];
        for (int i = 0; i < 256; i++) ident[i] = (uint8_t)i;
        NV_CUDA(cudaMemcpy(c->d_lut + 256, ident, 256, cudaMemcpyHostToDevice));     // identity LUT
        c->slots = new PlanSlot[NV_PLAN_SLOTS];
        c->ps = &c->slots[0];
        for (int i = 0; i < NV_PLAN_SLOTS; i++) NV_CUDA(cudaMalloc(&c->slots[i].d_plan, sizeof(PlanDev)));
        NV_CUDA(cudaMalloc(&c->d_counters, 16 * sizeof(int)));
        NV_CUDA(cudaMemset(c->d_counters, 0, 16 * sizeof(int)));     // from here on the grouping kernel leaves them at zero
        NV_CUDA(cudaMalloc(&c->d_deepq, NV_DEEPQ_CAP * sizeof(uint2)));
        return alloc_candidates(c, CAND_CAP, true);
    }();
    if (rc != NV_OK) { nv_ctx_destroy(c); return rc; }
    *out = c;
    return NV_OK;
}

static void batch_free(nv_ctx::Batch &b);

extern "C" void nv_ctx_destroy(nv_ctx *c)
{
    if (!c) return;
    cudaSetDevice(c->gpu);
    if (c->stream) cudaStreamSynchronize(c->stream);
    cudaFreeHost(c->h_frame); cudaFree(c->d_frame); cudaFree(c->d_gray); cudaFree(c->d_hist); cudaFree(c->d_lut);
    cudaFree(c->d_aux); for (auto &e : c->rtabs) cudaFree(e.d); cudaFree(c->d_sum);
    if (c->slots) {
        for (int i = 0; i < NV_PLAN_SLOTS; i++) {
            PlanSlot &sl = c->slots[i];
            cudaFree(sl.d_plan); cudaFree(sl.d_ptab); cudaFree(sl.d_maps);
            if (sl.dexec) cudaGraphExecDestroy(sl.dexec);
        }
        delete[] c->slots;
    }
    cudaFree(c->d_sq); cudaFree(c->d_pyr); cudaFree(c->d_tilt); cudaFree(c->d_vnf); cudaFree(c->d_depth);
    cudaFree(c->d_bits_ok); cudaFree(c->d_queue); cudaFree(c->d_queue2); cudaFree(c->d_deepq); cudaFree(c->d_counters); cudaFree(c->d_cand);
    cudaFree(c->d_cand_sorted); cudaFree(c->d_cand_rects); cudaFree(c->d_adj); cudaFree(c->d_result);
    cudaFree(c->d_cand_w); cudaFree(c->d_cls_wmax);
    cudaFreeHost(c->h_result);
    cudaFree(c->d_trk_prev); cudaFree(c->d_trk_hist); cudaFree(c->d_trk_scratch); cudaFreeHost(c->h_trk);
    if (c->gexec) cudaGraphExecDestroy(c->gexec);
    if (c->bexec) cudaGraphExecDestroy(c->bexec);
    batch_free(c->b);
    if (c->ev_done) cudaEventDestroy(c->ev_done);
    for (int i = 0; i < 2; i++) { if (c->ev_fork[i]) cudaEventDestroy(c->ev_fork[i]); if (c->ev_join[i]) cudaEventDestroy(c->ev_join[i]); }
    if (c->stream2) cudaStreamDestroy(c->stream2);
    for (int i = 0; i <= NV_NUM_STAGES; i++) if (c->prof_ev[i]) cudaEventDestroy(c->prof_ev[i]);
    if (c->stream) cudaStreamDestroy(c->stream);
    cudaGetLastError();
    delete c;
}

extern "C" int nv_ctx_set_scores(nv_ctx *ctx, int on)
{
    if (!ctx) { nv_set_error("null ctx"); return NV_ERR_ARG; }
    ctx->scores = on ? 1 : 0;
    return NV_OK;
}

// scores of the last collected call, parallel to its rectangles (result block: rects | weights | neighbour counts)
extern "C" int nv_get_scores(nv_ctx *ctx, int *neighbors, double *level_weights, int cap, int *n)
{
    if (!ctx) { nv_set_error("null ctx"); return NV_ERR_ARG; }
    if (!ctx->scores_ready || ctx->batch_last) { nv_set_error("no collected call with scores on"); return NV_ERR_STATE; }
    const int total = reinterpret_cast<const ResultHeader *>(ctx->h_result)->n_out, m = std::min(total, std::max(cap, 0));
    const uint8_t *w = ctx->h_result + sizeof(ResultHeader) + (size_t)ctx->result_cap * sizeof(nv_rect);
    const uint8_t *nb = w + (size_t)ctx->result_cap * sizeof(double);
    if (level_weights && m > 0) memcpy(level_weights, w, (size_t)m * sizeof(double));
    if (neighbors && m > 0) memcpy(neighbors, nb, (size_t)m * sizeof(int));
    if (n) *n = m;
    if (total > cap) { nv_set_error("%d rectangles, caller capacity %d", total, cap); return NV_ERR_CAPACITY; }
    return NV_OK;
}

extern "C" int nv_ctx_set_debug(nv_ctx *ctx, int debug)
{
    if (!ctx) { nv_set_error("null ctx"); return NV_ERR_ARG; }
    ctx->debug = debug ? 1 : 0;
    ctx->epoch++;
    for (int i = 0; ctx->slots && i < NV_PLAN_SLOTS; i++) ctx->slots[i].plan_valid = false;      // debug buffers are sized with the plan
    return NV_OK;
}

// ------------------------------------------------------------------------------------------------
// device-side timing
// ------------------------------------------------------------------------------------------------
static const char *k_stage_names[NV_NUM_STAGES] = {"face_prep", "hist_lut", "pyramid_rowscan", "integral_colscan",
                                                   "cascade_stage0", "cascade_tiles", "cascade_tail", "group_rectangles"};
extern "C" const char *nv_stage_name(int slot) { return slot >= 0 && slot < NV_NUM_STAGES ? k_stage_names[slot] : ""; }

static inline void prof_mark(nv_ctx *ctx, int idx)
{
    if (!ctx->profile) return;
    // inside a stream capture the record becomes an event-record NODE of the graph (cudaEventRecordExternal), so that
    // the stage times can be read after every replay
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(ctx->stream, &cs);
    if (cs == cudaStreamCaptureStatusActive) cudaEventRecordWithFlags(ctx->prof_ev[idx], ctx->stream, cudaEventRecordExternal);
    else cudaEventRecord(ctx->prof_ev[idx], ctx->stream);
    ctx->prof_set[idx] = true;
}

extern "C" int nv_ctx_set_profile(nv_ctx *ctx, int on)
{
    if (!ctx) { nv_set_error("null ctx"); return NV_ERR_ARG; }
    NV_CUDA(cudaSetDevice(ctx->gpu));
    if (on && !ctx->prof_ev[0])
        for (int i = 0; i <= NV_NUM_STAGES; i++) NV_CUDA(cudaEventCreate(&ctx->prof_ev[i]));
    if (ctx->profile != (on ? 1 : 0)) ctx->epoch++;       // graphs are captured with or without the event-record nodes
    ctx->profile = on ? 1 : 0;
    return NV_OK;
}

extern "C" int nv_ctx_get_stage_times(nv_ctx *ctx, float *ms, int cap, int *n)
{
    if (!ctx || !ms) { nv_set_error("null argument"); return NV_ERR_ARG; }
    if (!ctx->profile || ctx->pending) { nv_set_error("profiling off or call still pending"); return NV_ERR_STATE; }
    if (ctx->batch_last) { nv_set_error("stage times describe single calls: the last call was a batch"); return NV_ERR_STATE; }
    NV_CUDA(cudaSetDevice(ctx->gpu));
    int m = std::min(cap, NV_NUM_STAGES);
    for (int i = 0; i < m; i++) {
        ms[i] = 0.f;
        if (ctx->prof_set[i] && ctx->prof_set[i + 1]) NV_CUDA(cudaEventElapsedTime(&ms[i], ctx->prof_ev[i], ctx->prof_ev[i + 1]));
    }
    if (n) *n = m;
    return NV_OK;
}

extern "C" int nv_event_create(void **ev)
{
    if (!ev) { nv_set_error("null argument"); return NV_ERR_ARG; }
    cudaEvent_t e;
    NV_CUDA(cudaEventCreate(&e));
    *ev = e;
    return NV_OK;
}
extern "C" int nv_event_record(nv_ctx *ctx, void *ev)
{
    if (!ctx || !ev) { nv_set_error("null argument"); return NV_ERR_ARG; }
    NV_CUDA(cudaSetDevice(ctx->gpu));
    NV_CUDA(cudaEventRecord((cudaEvent_t)ev, ctx->stream));
    return NV_OK;
}
extern "C" int nv_event_elapsed_ms(void *e0, void *e1, float *ms)
{
    if (!e0 || !e1 || !ms) { nv_set_error("null argument"); return NV_ERR_ARG; }
    NV_CUDA(cudaEventSynchronize((cudaEvent_t)e1));
    NV_CUDA(cudaEventElapsedTime(ms, (cudaEvent_t)e0, (cudaEvent_t)e1));
    return NV_OK;
}
extern "C" void nv_event_destroy(void *ev) { if (ev) cudaEventDestroy((cudaEvent_t)ev); }

// ------------------------------------------------------------------------------------------------
// plan: scale list, level geometry (SURVEY.md A.4 + the oracle's probes), coefficient tables
// ------------------------------------------------------------------------------------------------
static inline int cv_round(double v) { return (int)lrint(v); }
static inline int cv_roundf(float v) { return (int)lrintf(v); }
static inline int align_up(int v, int a) { return (v + a - 1) / a * a; }

// INTER_LINEAR_EXACT coefficients (8 fractional bits), branch-free for the kernel: entry = (i, f) means
// 256 * value = src[i] * (256 - f) + src[i + 1] * f with i + 1 < ssize ALWAYS — the clamped ends, where OpenCV takes a
// single source sample, are written as (0, 0) and (ssize - 2, 256).  `lead` dummy entries (0, 0) come first (the row
// kernel indexes the x table by integral column c = x + 1), `total` entries are written in all.
static void exact_coefs(int ssize, int dsize, int2 *tab, int lead, int total)
{
    double scale = 1.0 / ((double)dsize / ssize);
    for (int k = 0; k < total; k++) tab[k] = make_int2(0, 0);
    for (int d = 0; d < dsize; d++) {
        double f = scale * (d + 0.5) - 0.5;
        int i = (int)floor(f);
        if (i >= 0 && i < ssize - 1) tab[lead + d] = make_int2(i, cv_round((f - i) * 256.0));
        else if (i < 0) tab[lead + d] = make_int2(0, 0);
        else tab[lead + d] = ssize >= 2 ? make_int2(ssize - 2, 256) : make_int2(0, 0);
    }
}

static int ensure_plan(nv_ctx *ctx, const nv_cascade *casc, int W, int H, const nv_detect_params *p)
{
    if (!(p->scale_factor > 1.0)) {
        nv_set_error("scale_factor must be > 1 (got %g): OpenCV would never terminate", p->scale_factor);
        return NV_ERR_ARG;
    }
    PlanKey key;
    key.W = W; key.H = H; key.win_w = casc->h.win_w; key.win_h = casc->h.win_h;
    key.min_w = p->min_w; key.min_h = p->min_h; key.max_w = p->max_w; key.max_h = p->max_h; key.sf = p->scale_factor;
    key.casc = casc->uid;
    if (ctx->ps->plan_valid && key == ctx->ps->pkey) { ctx->ps->last_use = ++ctx->use_clock; return NV_OK; }
    // another cached plan?  (nested ROI stages: the same few ROI sizes come back frame after frame)
    PlanSlot *victim = nullptr;
    for (int i = 0; i < NV_PLAN_SLOTS; i++) {
        PlanSlot &sl = ctx->slots[i];
        if (sl.plan_valid && key == sl.pkey) {
            ctx->ps = &sl;
            sl.last_use = ++ctx->use_clock;
            if (sl.buf_gen != ctx->buf_gen) { sl.tp_casc = 0; sl.buf_gen = ctx->buf_gen; }   // its tensor maps point into freed buffers
            return NV_OK;
        }
        if (!victim || (!sl.plan_valid && victim->plan_valid) || (sl.plan_valid == victim->plan_valid && sl.last_use < victim->last_use))
            victim = &sl;
    }
    ctx->ps = victim;
    ctx->ps->plan_valid = false;
    ctx->ps->last_use = ++ctx->use_clock;

    PlanDev &P = ctx->ps->plan;
    memset(&P, 0, sizeof P);
    P.W = W; P.H = H; P.win_w = key.win_w; P.win_h = key.win_h;
    int max_w = p->max_w, max_h = p->max_h;
    if (max_w == 0 || max_h == 0) { max_w = W; max_h = H; }
    std::vector<float> scales;
    for (double f = 1;; f *= p->scale_factor) {
        int ww = cv_round(key.win_w * f), wh = cv_round(key.win_h * f);
        if (ww > max_w || wh > max_h || ww > W || wh > H) break;
        if (ww < p->min_w || wh < p->min_h) continue;
        scales.push_back((float)f);
        if (scales.size() > 4096) break;
    }
    int nstripes = 1;
    long long iofs = 0, wofs = 0, bofs = 0, tofs = 0, pofs = 0;
    int nl = 0;
    for (size_t k = 0; k < scales.size(); k++) {
        float sc = scales[k];
        int lw = cv_roundf((float)W / sc), lh = cv_roundf((float)H / sc);       // float division, as OpenCV
        int rx = lw + 1 - key.win_w, ry = lh + 1 - key.win_h;
        if (k == 0) nstripes = std::max((std::max(rx, 0) + 31) / 32, 1);
        if (rx <= 0 || ry <= 0) continue;
        int ystep = sc >= 2.f ? 1 : 2;
        // stripe split of detectMultiScale: the last stripe is clamped, an odd tail row may be lost
        int stripe = std::max((ry / ystep + nstripes - 1) / nstripes, 1) * ystep;
        long long lim = (long long)stripe * nstripes;
        if (lim < ry) ry = (int)lim;
        if (nl >= NV_MAX_LEVELS) { nv_set_error("more than %d pyramid levels", NV_MAX_LEVELS); return NV_ERR_CAPACITY; }
        LevelDesc &L = P.lv[nl++];
        L.scale = sc; L.lw = lw; L.lh = lh; L.ystep = ystep;
        L.nx = (rx + ystep - 1) / ystep; L.ny = (ry + ystep - 1) / ystep; L.nxw = (L.nx + 31) / 32;
        if (L.nx > 8191 || L.ny > 8191) { nv_set_error("level too large for 13-bit window ids"); return NV_ERR_CAPACITY; }
        L.iplane = align_up((lw + 1 + ystep - 1) / ystep, 4);
        L.ipitch = L.iplane * ystep;
        L.iofs = (int)iofs; iofs += (long long)L.ipitch * (lh + 1);
        L.wofs = (int)wofs; wofs += (long long)L.nx * L.ny;
        L.bofs = (int)bofs; bofs += (long long)L.nxw * L.ny;
        // x table: indexed by integral column (one leading dummy), padded to whole groups of four entries; both tables 16-byte aligned
        L.xtab = (int)tofs; L.ytab = (int)tofs + align_up(lw + 1, 4); tofs += align_up(lw + 1, 4) + align_up(lh, 2);
        L.pofs = (int)pofs; pofs += (long long)lw * lh;
        L.rowblk0 = P.total_rowblk; P.total_rowblk += (lh + 7) / 8;
        L.colblk0 = P.total_colblk; P.total_colblk += (L.ipitch + NV_COLBLK - 1) / NV_COLBLK;
        L.chunk0 = P.total_chunks; P.total_chunks += L.nxw * L.ny;
        L.row0 = P.total_rows; P.total_rows += L.ny;
        L.dblk0 = P.total_dblk; P.total_dblk += (lw + lh + 255) / 256;
        L.cntx = (L.nx + NV_CTX - 1) / NV_CTX;
        int cnt = L.cntx * ((L.ny + NV_CTY - 1) / NV_CTY);
        if (ystep == 2) { L.ctile0 = P.ctiles2; P.ctiles2 += cnt; P.nlv2 = nl; }
        else { L.ctile0 = P.ctiles1; P.ctiles1 += cnt; }
        L.wtile0 = 0; L.wntx = 0;
        if (ystep == 1) {
            L.wntx = (L.nx + NV_WTX - 1) / NV_WTX;
            L.wtile0 = P.wtiles[1]; P.wtiles[1] += L.wntx * ((L.ny + NV_WTY - 1) / NV_WTY);
        }
        if (iofs > 0x7fffffffLL || wofs > 0x7fffffffLL) { nv_set_error("frame too large"); return NV_ERR_CAPACITY; }
    }
    P.nlevels = nl;
    P.total_windows = (int)wofs;

    NV_CUDA(cudaStreamSynchronize(ctx->stream));      // previous frame may still read the old plan
    if (nl > 0) {
        std::vector<int2> tab((size_t)tofs);
        for (int l = 0; l < nl; l++) {
            exact_coefs(W, P.lv[l].lw, &tab[P.lv[l].xtab], 1, align_up(P.lv[l].lw + 1, 4));
            exact_coefs(H, P.lv[l].lh, &tab[P.lv[l].ytab], 0, align_up(P.lv[l].lh, 2));
        }
        int rc;
        if ((rc = ensure(&ctx->ps->d_ptab, &ctx->ps->ptab_cap, (size_t)tofs * 2)) != NV_OK) return rc;
        NV_CUDA(cudaMemcpy(ctx->ps->d_ptab, tab.data(), (size_t)tofs * sizeof(int2), cudaMemcpyHostToDevice));
        const void *old[8] = {ctx->d_sum, ctx->d_sq, ctx->d_vnf, ctx->d_queue, ctx->d_bits_ok, ctx->d_depth, ctx->d_pyr, ctx->d_tilt};
        // on EVERY way out of this block — a failed allocation included — cached tensor maps and graphs of the other plan
        // slots are invalidated if a shared buffer was freed or moved
        struct MovedGuard {
            nv_ctx *c; const void *const *old;
            ~MovedGuard()
            {
                const void *now[8] = {c->d_sum, c->d_sq, c->d_vnf, c->d_queue, c->d_bits_ok, c->d_depth, c->d_pyr, c->d_tilt};
                if (memcmp(old, now, sizeof now)) { c->buf_gen++; c->epoch++; }
            }
        } moved_guard{ctx, old};
        size_t icap = ctx->integ_cap;
        if ((rc = ensure(&ctx->d_sum, &icap, (size_t)iofs, true)) != NV_OK) return rc;
        if ((rc = ensure(&ctx->d_sq, &ctx->integ_cap, (size_t)iofs, true)) != NV_OK) return rc;
        size_t wcap = ctx->win_cap;
        if ((rc = ensure(&ctx->d_vnf, &wcap, (size_t)wofs)) != NV_OK) return rc;
        if ((rc = ensure(&ctx->d_queue, &ctx->queue_cap, (size_t)wofs)) != NV_OK) return rc;
        ctx->win_cap = wcap;
        // three bit planes of `bofs` words each: alive after stage 0 and the skip rule | failed stage 0 | valid and passed the variance test
        if ((rc = ensure(&ctx->d_bits_ok, &ctx->bits_cap, (size_t)bofs * 3)) != NV_OK) return rc;
        ctx->ps->bits_words = bofs;
        if (ctx->debug) {
            if ((rc = ensure(&ctx->d_depth, &ctx->depth_cap, (size_t)wofs)) != NV_OK) return rc;
            if ((rc = ensure(&ctx->d_pyr, &ctx->pyr_cap, (size_t)pofs)) != NV_OK) return rc;
        }
        if (ctx->need_tilt && (rc = ensure(&ctx->d_tilt, &ctx->tilt_cap, ctx->integ_cap)) != NV_OK) return rc;
        ctx->ps->max_lw = 0;
        for (int l = 0; l < nl; l++) ctx->ps->max_lw = std::max(ctx->ps->max_lw, P.lv[l].lw);
    }
    NV_CUDA(cudaMemcpy(ctx->ps->d_plan, &P, sizeof(PlanDev), cudaMemcpyHostToDevice));
    ctx->ps->pkey = key;
    ctx->ps->plan_valid = true;
    ctx->ps->tp_casc = 0;                  // tensor maps and tile geometry follow the plan
    ctx->ps->buf_gen = ctx->buf_gen;
    ctx->ps->gen++;
    if (ctx->ps->dexec) { cudaGraphExecDestroy(ctx->ps->dexec); ctx->ps->dexec = nullptr; }
    ctx->ps->dkey = DetGraphKey(); ctx->ps->dkey_seen = DetGraphKey();
    return NV_OK;
}

// ---- tile-kernel parameters: tensor maps over each level's sum integral + bulk-stage classifiers ----
typedef CUresult (*encode_tiled_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                    const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static encode_tiled_fn get_encode_tiled()
{
    static encode_tiled_fn fn = []() -> encode_tiled_fn {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess) { cudaGetLastError(); return nullptr; }
        return (encode_tiled_fn)p;
    }();
    return fn;
}

static int ensure_tile_params(nv_ctx *ctx, const nv_cascade *casc)
{
    if (ctx->ps->tp_casc == casc->uid) return NV_OK;
    const PlanDev &P = ctx->ps->plan;
    const DevCascade &m = casc->meta;
    ctx->ps->tp_casc = casc->uid;
    ctx->ps->use_tiles = false;  ctx->ps->use_s0t = false;
    ctx->ps->gen++;                                              // graphs hold the parameter banks by value
    if (ctx->ps->dexec) { cudaGraphExecDestroy(ctx->ps->dexec); ctx->ps->dexec = nullptr; }
    ctx->ps->use_s0p = !casc->h.general && P.nlevels > 0 && fill_stage0_params(casc, P, &ctx->ps->s0p);
    encode_tiled_fn enc = get_encode_tiled();
    if (casc->h.general || !enc || m.win_w > 32 || m.win_h > 32 || P.nlevels == 0) return NV_OK;
    // bulk stages: as many as fit the parameter bank
    int end = 1;
    while (end < m.nstages && end < NV_BULK_MAX_STAGES && m.stage_first[end + 1] - m.stage_first[1] <= NV_BULK_MAX_STUMPS) end++;
    ctx->ps->bulk_end = end;
    static_assert(sizeof(CUtensorMap) == 128, "tensor map size");
    // maps[l]: the bulk kernel's box of level l; maps[NV_MAX_LEVELS + l]: the 64x32-window box of the dense stage-0 kernel
    // (the same box unless the level's bulk stages run on wide tiles)
    alignas(64) CUtensorMap maps[2 * NV_MAX_LEVELS];
    memset(maps, 0, sizeof maps);
    if (!ctx->ps->d_maps) NV_CUDA(cudaMalloc(&ctx->ps->d_maps, sizeof maps));
    for (int c = 0; c < 2; c++) {
        int ys = c == 0 ? 2 : 1;
        TileParams &tp = ctx->ps->tp[c];
        // tile geometry for tw x th windows.  Columns per plane: the pitch is 4 (mod 8) words, so that the bank class
        // (lx + kskew * ly) & 31 of a window moves by a multiple of 4 that is not a multiple of 32 from one window row to
        // the next
        struct Geo { int cp, rt, ps, kskew; };
        auto geometry = [&](int tw, int th) {
            Geo g;
            g.cp = align_up(tw + (ys == 2 ? m.win_w / 2 : m.win_w) + 1, 4);
            if (g.cp % 8 == 0) g.cp += 4;
            g.rt = (th - 1) * ys + m.win_h + 1;
            g.kskew = (ys * g.cp) & 31;
            g.ps = align_up(g.rt * g.cp, 32);
            return g;
        };
        const Geo g0 = geometry(NV_CTX, NV_CTY);
        const Geo g = ys == 1 ? geometry(NV_WTX, NV_WTY) : g0;
        if (g.cp > 256 || g.rt > 256) return NV_OK;             // TMA box limit: keep the generic queue path
        tp.cp = g.cp; tp.rt = g.rt; tp.kskew = g.kskew; tp.ps = g.ps;
        tp.level_begin = c == 0 ? 0 : P.nlv2;
        tp.level_end = c == 0 ? P.nlv2 : P.nlevels;
        fill_bulk_stumps(casc, ys, tp.cp, tp.ps, 1, end, &tp);
        Stage0TileParams &s0 = ctx->ps->s0t[c];
        const bool s0ok = tp.fast && fill_stage0_tile_params(casc, ys, g0.cp, g0.rt, g0.ps, g0.kskew, &s0);
        ctx->ps->use_s0t = c == 0 ? s0ok : (ctx->ps->use_s0t && s0ok);
        s0.level_begin = tp.level_begin; s0.level_end = tp.level_end;
        for (int l = tp.level_begin; l < tp.level_end; l++) {
            const LevelDesc &L = P.lv[l];
            cuuint64_t gdim[2] = {(cuuint64_t)L.ipitch, (cuuint64_t)(L.lh + 1)};
            cuuint64_t gstr[1] = {(cuuint64_t)L.ipitch * 4};
            cuuint32_t estr[2] = {1, 1};
            for (int k = 0; k < 2; k++) {
                cuuint32_t box[2] = {(cuuint32_t)(k == 0 ? g.cp : g0.cp), (cuuint32_t)(k == 0 ? g.rt : g0.rt)};
                CUresult r = enc(&maps[k * NV_MAX_LEVELS + l], CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, ctx->d_sum + L.iofs, gdim, gstr, box, estr,
                                 CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                 CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
                if (r != CUDA_SUCCESS) return NV_OK;   // keep the generic queue path for this plan
            }
        }
    }
    NV_CUDA(cudaStreamSynchronize(ctx->stream));
    NV_CUDA(cudaMemcpy(ctx->ps->d_maps, maps, sizeof maps, cudaMemcpyHostToDevice));
    ctx->ps->use_tiles = true;
    return NV_OK;
}

// ------------------------------------------------------------------------------------------------
// detectMultiScale on a device-resident gray image (+ LUT), everything stream-ordered
// ------------------------------------------------------------------------------------------------
// host-side preparation (may allocate, copy tables and synchronise): plan, cascade upload, tile parameters
static int detect_prepare(nv_ctx *ctx, nv_cascade *casc, int W, int H, const nv_detect_params *p)
{
    int rc = ensure_plan(ctx, casc, W, H, p);
    if (rc != NV_OK) return rc;
    if ((rc = cascade_on_device(casc, ctx->gpu, ctx->stream, &ctx->cur_stumps, &ctx->cur_meta)) != NV_OK) return rc;
    ctx->cur_tail = nullptr; ctx->cur_tail_base = nullptr;
    ctx->use_gen = casc->h.general != 0;
    if (ctx->use_gen) {
        std::lock_guard<std::mutex> lk(casc->mu);
        ctx->cur_gen = casc->d_gen[ctx->gpu];
    }
    ctx->cur_tilted = casc->h.has_tilted != 0;
    if (ctx->cur_tilted) {
        // the tilted integral is allocated when the first cascade with tilted features shows up (and kept: the eye
        // element alternates between an upright face model and tilted eye models)
        if (!ctx->need_tilt || ctx->tilt_cap < ctx->integ_cap) {
            NV_CUDA(cudaStreamSynchronize(ctx->stream));
            ctx->need_tilt = true;
            if ((rc = ensure(&ctx->d_tilt, &ctx->tilt_cap, ctx->integ_cap)) != NV_OK) return rc;
            ctx->epoch++; ctx->buf_gen++;
        }
    }
    if (casc->tail_fast) {
        std::lock_guard<std::mutex> lk(casc->mu);
        ctx->cur_tail = casc->d_tail[ctx->gpu]; ctx->cur_tail_base = casc->d_tail_base[ctx->gpu];
    }
    if (ctx->use_gen && ctx->ps->plan.total_windows > NV_SMALL_PLAN_WINDOWS && ctx->queue2_cap < ctx->queue_cap) {
        // a tree / tilted model over a large image compacts its survivors between stage ranges: second queue, same size
        NV_CUDA(cudaStreamSynchronize(ctx->stream));
        if ((rc = ensure(&ctx->d_queue2, &ctx->queue2_cap, ctx->queue_cap)) != NV_OK) return rc;
        ctx->epoch++; ctx->buf_gen++;
    }
    if ((rc = ensure_tile_params(ctx, casc)) != NV_OK) return rc;
    if (p->min_neighbors > 0 && ctx->adj_cap < (size_t)ctx->cand_cap) {      // grown earlier for an ungrouped call
        NV_CUDA(cudaStreamSynchronize(ctx->stream));
        if ((rc = alloc_candidates(ctx, std::min(ctx->cand_cap, CAND_CAP_GROUPED), true)) != NV_OK) return rc;
    }
    return NV_OK;
}

// the stream-ordered part: only asynchronous work on ctx->stream, so it can be captured into a CUDA graph
static int detect_enqueue(nv_ctx *ctx, nv_cascade *casc, const uint8_t *d_gray, int W, int H, int gstride,
                          const uint8_t *d_lut, const nv_detect_params *p, int *nlaunch)
{
    const DevStump *stumps = ctx->cur_stumps;
    const DevCascade *meta = ctx->cur_meta;
    const PlanDev &P = ctx->ps->plan;
    cudaStream_t st = ctx->stream;
    int nl = 0;
    for (int i = 2; i <= NV_NUM_STAGES; i++) ctx->prof_set[i] = false;
    // (no memset of the counters here: the last kernel of every call, k_group / k_group_fused, zeroes them when it has read
    // them — a memset node cost a small call more than any of its kernels' launch gaps.  Should a launch in between fail, that
    // kernel never runs: the guard clears them on the way out, best effort.)
    struct CountersGuard {
        nv_ctx *c; cudaStream_t s; bool done = false;
        ~CountersGuard() { if (!done) { cudaMemsetAsync(c->d_counters, 0, 16 * sizeof(int), s); cudaGetLastError(); } }
    } counters_guard{ctx, st};
    if (P.nlevels > 0) {
        int16_t *depth = ctx->debug ? ctx->d_depth : nullptr;
        prof_mark(ctx, 2);
        const uint32_t *tilt = ctx->use_gen && ctx->cur_tilted ? ctx->d_tilt : nullptr;
        NV_CUDA(launch_pyr_rowscan(ctx->ps->d_plan, P.total_rowblk, d_gray, gstride, d_lut, ctx->ps->d_ptab, ctx->d_sum, ctx->d_sq,
                                   ctx->debug ? ctx->d_pyr : nullptr, st));
        prof_mark(ctx, 3);
        NV_CUDA(launch_colscan(ctx->ps->d_plan, P.total_colblk, ctx->d_sum, ctx->d_sq, st));
        if (tilt) { NV_CUDA(launch_tilted(ctx->ps->d_plan, P.total_dblk, ctx->d_sum, ctx->d_tilt, st)); nl += 2; }
        prof_mark(ctx, 4);
        // small plan of a cascade with the certificates: every window alive after stage 0 goes to the warp-per-window kernel;
        // k_stage0_rows_p appends them to its queue itself
        const bool small_fast = ctx->ps->use_tiles && ctx->cur_tail && P.total_windows <= NV_SMALL_PLAN_WINDOWS && casc->meta.nstages > 1;
        const int qcap = (int)std::min<size_t>(ctx->queue_cap, 0x7fffffff);
        bool queued = false;
        if (ctx->use_gen) {
            NV_CUDA(launch_stage0_rows_gen(ctx->ps->d_plan, P.total_rows, meta, ctx->cur_gen, ctx->d_sum, ctx->d_sq, tilt, ctx->d_vnf,
                                           ctx->d_bits_ok, ctx->d_counters, depth, st));
        } else if (ctx->ps->use_tiles && ctx->ps->use_s0t && P.total_windows > NV_SMALL_PLAN_WINDOWS) {
            // large plan, FAST cascade: stage 0 densely on the bulk kernel's tiles, then the skip rule along the rows
            uint32_t *bits_fail = ctx->d_bits_ok + ctx->ps->bits_words, *bits_okv = ctx->d_bits_ok + 2 * (size_t)ctx->ps->bits_words;
            const bool fork = P.ctiles2 > 0 && P.ctiles1 > 0;      // the ystep-1 levels' launch goes to the side stream
            if (fork) { NV_CUDA(cudaEventRecord(ctx->ev_fork[0], st)); NV_CUDA(cudaStreamWaitEvent(ctx->stream2, ctx->ev_fork[0], 0)); }
            for (int c = 0; c < 2; c++) {
                Stage0TileParams &s0 = ctx->ps->s0t[c];
                int ntiles = c == 0 ? P.ctiles2 : P.ctiles1;
                if (ntiles == 0) continue;
                s0.maps = ctx->ps->d_maps + NV_MAX_LEVELS; s0.plan = ctx->ps->d_plan; s0.sq = ctx->d_sq; s0.vnf = ctx->d_vnf;
                s0.bits_fail = bits_fail; s0.bits_okv = bits_okv;
                NV_CUDA(launch_stage0_tiles(s0, c == 0 ? 2 : 1, ntiles, c == 1 && fork ? ctx->stream2 : st));
                nl++;
            }
            if (fork) { NV_CUDA(cudaEventRecord(ctx->ev_join[0], ctx->stream2)); NV_CUDA(cudaStreamWaitEvent(st, ctx->ev_join[0], 0)); }
            NV_CUDA(launch_stage0_chain(P, bits_fail, bits_okv, ctx->d_bits_ok, ctx->d_counters, depth, st));
        } else if (ctx->ps->use_s0p) {
            Stage0Params &sp = ctx->ps->s0p;
            sp.sum = ctx->d_sum; sp.sq = ctx->d_sq; sp.vnf = ctx->d_vnf; sp.bits_alive = ctx->d_bits_ok;
            sp.counters = ctx->d_counters; sp.depth = depth;
            sp.queue = small_fast ? ctx->d_queue : nullptr; sp.queue_cap = qcap; sp.queue_cidx = 3;
            queued = small_fast;
            NV_CUDA(launch_stage0_rows_p(sp, st));
        } else
            NV_CUDA(launch_stage0_rows(ctx->ps->d_plan, P.total_rows, meta, stumps, ctx->d_sum, ctx->d_sq, ctx->d_vnf,
                                       ctx->d_bits_ok, ctx->d_counters, depth, st));
        prof_mark(ctx, 5);
        nl += 3;
        if (small_fast) {
            // small plan: every window alive after stage 0 goes straight to the warp-per-window kernel (same exactness
            // certificates as the tail it normally is, nv_cascade::tail_fast)
            if (!queued) {
                NV_CUDA(launch_alive_to_queue(ctx->ps->d_plan, P.total_rows, ctx->d_vnf, ctx->d_bits_ok, ctx->d_queue, ctx->d_counters,
                                              qcap, st, 3));
                nl++;
            }
            prof_mark(ctx, 6);
            // stages narrower than NV_TAIL_BLOCK_MIN_STUMPS with a warp per window, the deep ones with a block per window —
            // unless the whole classifier table fits shared memory: then k_cascade_tail_tab takes every stage (measured,
            // profiles/r2_summary.md section 8: a 96x64 ROI detect 100.6 -> 88.5 us per call, eyes-in-faces 374 -> 359 us)
            int split = 1;
            while (split < casc->meta.nstages && casc->meta.stage_first[split + 1] - casc->meta.stage_first[split] < NV_TAIL_BLOCK_MIN_STUMPS) split++;
            if (tail_tab_smem(casc->meta, 1, casc->meta.nstages) <= NV_TAILTAB_MAX_SMEM) split = casc->meta.nstages;
            if (tail_tab_smem(casc->meta, 1, split) <= NV_TAILTAB_MAX_SMEM)
                NV_CUDA(launch_cascade_tail_tab(ctx->ps->d_plan, meta, casc->meta, ctx->cur_tail, ctx->cur_tail_base, ctx->d_sum, ctx->d_queue,
                                                ctx->d_counters, ctx->d_cand, ctx->cand_cap, depth, 1, split, ctx->d_deepq, NV_DEEPQ_CAP, st));
            else
                NV_CUDA(launch_cascade_tail_fast(ctx->ps->d_plan, meta, ctx->cur_tail, ctx->cur_tail_base, ctx->d_sum, ctx->d_queue,
                                                 ctx->d_counters, ctx->d_cand, ctx->cand_cap, depth, 1, split, ctx->d_deepq, NV_DEEPQ_CAP, st,
                                                 8 * (casc->meta.win_w + 1) * (casc->meta.win_h + 1) * 4));
            nl += 1;
            if (split < casc->meta.nstages) {
                NV_CUDA(launch_cascade_tail_block(ctx->ps->d_plan, meta, ctx->cur_tail, ctx->cur_tail_base, ctx->d_sum, ctx->d_deepq,
                                                  ctx->d_counters, 6, ctx->d_cand, ctx->cand_cap, depth, split, -1, st));
                nl++;
            }
        } else if (ctx->ps->use_tiles) {
            const bool fork = P.ctiles2 > 0 && P.ctiles1 > 0;
            if (fork) { NV_CUDA(cudaEventRecord(ctx->ev_fork[1], st)); NV_CUDA(cudaStreamWaitEvent(ctx->stream2, ctx->ev_fork[1], 0)); }
            // Launch order decides what the two kernels share.  The ystep-2 levels first: their 742 blocks fill every SM's
            // shared memory and the wide blocks of the ystep-1 levels follow as they drain — 2970 frames/s with eight frames
            // in flight, bulk stages 0.34 ms when a frame is alone.  The ystep-1 levels first was measured: their 368 wide
            // blocks leave room for a block of the other kernel on every SM, so a lone frame's bulk stages take 0.27 ms, but
            // eight frames in flight lose 4 % (2845 frames/s).
            for (int c = 0; c < 2; c++) {
                TileParams &tp = ctx->ps->tp[c];
                const cudaStream_t cst = c == 1 && fork ? ctx->stream2 : st;
                if ((c == 0 ? P.ctiles2 : P.ctiles1) == 0) continue;
                tp.plan = ctx->ps->d_plan; tp.bits_alive = ctx->d_bits_ok; tp.vnf = ctx->d_vnf; tp.depth = depth;
                tp.tail = ctx->d_queue; tp.cand = ctx->d_cand; tp.counters = ctx->d_counters; tp.maps = ctx->ps->d_maps;
                tp.tail_cap = qcap; tp.cand_cap = ctx->cand_cap;
                if (c == 0) NV_CUDA(launch_cascade_classes(tp, P.ctiles2, cst));
                else NV_CUDA(launch_cascade_wide(tp, P.wtiles[1], cst));
                nl++;
            }
            if (fork) { NV_CUDA(cudaEventRecord(ctx->ev_join[1], ctx->stream2)); NV_CUDA(cudaStreamWaitEvent(st, ctx->ev_join[1], 0)); }
            prof_mark(ctx, 6);
            if (ctx->ps->bulk_end < casc->meta.nstages && ctx->cur_tail) {
                // the survivors of the bulk stages (~15 000 per config-3 frame, most of them gone within a few stages): a warp
                // per window.  (Handing the deep ones to the block-per-window kernel after four stages was measured: 55 us
                // against 45 us isolated, 2538 against 2577 frames/s — with that many windows the warp kernel is bound by
                // throughput, not by its deepest window; the split pays on small plans only.  Nor does k_cascade_tail_tab pay
                // here, profiles/r2_summary.md section 8: tail 45 -> 49 / 45 / 41 us with 8 / 16 / 32 warps per block, bench.py
                // -1 .. -4 % — fewer resident warps for these shallow windows, and 84 KB blocks queue behind the bulk kernels of
                // the other streams.)
                NV_CUDA(launch_cascade_tail_fast(ctx->ps->d_plan, meta, ctx->cur_tail, ctx->cur_tail_base, ctx->d_sum, ctx->d_queue,
                                                 ctx->d_counters, ctx->d_cand, ctx->cand_cap, depth, ctx->ps->bulk_end, casc->meta.nstages,
                                                 nullptr, qcap, st, 8 * (casc->meta.win_w + 1) * (casc->meta.win_h + 1) * 4));
                nl++;
            } else if (ctx->ps->bulk_end < casc->meta.nstages) {
                NV_CUDA(launch_cascade_tail(ctx->ps->d_plan, meta, stumps, ctx->d_sum, ctx->d_queue, ctx->d_counters, ctx->d_cand,
                                            ctx->cand_cap, depth, ctx->ps->bulk_end, casc->h.order_free, 148 * 8, st,
                                            8 * (casc->meta.win_w + 1) * (casc->meta.win_h + 1) * 4));
                nl++;
            }
        } else {
            NV_CUDA(launch_alive_to_queue(ctx->ps->d_plan, P.total_rows, ctx->d_vnf, ctx->d_bits_ok, ctx->d_queue, ctx->d_counters,
                                          qcap, st));
            prof_mark(ctx, 6);
            if (ctx->use_gen && P.total_windows > NV_SMALL_PLAN_WINDOWS && ctx->d_queue2 && ctx->queue2_cap >= ctx->queue_cap && casc->meta.nstages > 1) {
                int extra = 0;                                   // large plan: stage-wise compaction between thread-per-window passes
                NV_CUDA(launch_queue_stages_gen_staged(ctx->ps->d_plan, meta, ctx->cur_gen, ctx->d_sum, tilt, ctx->d_queue, ctx->d_queue2, qcap,
                                                       ctx->d_counters, ctx->d_cand, ctx->cand_cap, depth, casc->meta.nstages,
                                                       casc->h.order_free, st, &extra));
                nl += extra - 1;
            } else if (ctx->use_gen)
                NV_CUDA(launch_queue_stages_gen(ctx->ps->d_plan, meta, ctx->cur_gen, ctx->d_sum, tilt, ctx->d_queue, ctx->d_counters,
                                                ctx->d_cand, ctx->cand_cap, depth, 148 * 8, casc->h.order_free, st));
            else
                NV_CUDA(launch_queue_stages(ctx->ps->d_plan, meta, stumps, ctx->d_sum, ctx->d_queue, ctx->d_counters, ctx->d_cand,
                                            ctx->cand_cap, depth, 148 * 8, st));
            nl += 2;
        }
    }
    prof_mark(ctx, 7);
    const ScoreArgs sa = {ctx->cur_meta, ctx->cur_stumps, ctx->use_gen ? ctx->cur_gen : GenModel{}, ctx->use_gen ? 1 : 0, ctx->d_sum, ctx->d_sq,
                          ctx->use_gen && ctx->cur_tilted ? ctx->d_tilt : nullptr, ctx->d_cand_w, ctx->d_cls_wmax};
    // small plans: sort + similarity matrix + grouping in one launch of one block (k_group_fused).  The grouping kernel writes
    // header and rectangles into the page-locked result block itself (mapped memory, posted writes over PCIe, visible once
    // the stream has been waited for): no device-to-host copy behind it.
    NV_CUDA(launch_group(ctx->ps->d_plan, ctx->d_counters, ctx->d_cand, ctx->cand_cap, ctx->d_cand_sorted, ctx->d_cand_rects,
                         ctx->d_adj, ctx->d_grp, p->min_neighbors, 0.2, W, H, ctx->d_result, ctx->result_cap, 148 * 2, st, &nl,
                         P.total_windows <= NV_SMALL_PLAN_WINDOWS, ctx->h_result, ctx->scores ? &sa : nullptr));
    prof_mark(ctx, 8);
    *nlaunch += nl;
    counters_guard.done = true;
    return NV_OK;
}

static void detect_bookkeeping(nv_ctx *ctx, nv_cascade *casc, const uint8_t *d_gray, int W, int H, int gstride,
                               const uint8_t *d_lut, const nv_detect_params *p)
{
    ctx->last_min_neighbors = p->min_neighbors;
    ctx->last_casc = casc; ctx->last_params = *p; ctx->last_W = W; ctx->last_H = H;
    ctx->tap_gray = d_gray; ctx->tap_lut = d_lut; ctx->tap_stride = gstride;
    ctx->last_scores = ctx->scores != 0; ctx->scores_ready = false;
    ctx->pending = true;
    ctx->batch_last = false;
}

int nv_detect_device(nv_ctx *ctx, nv_cascade *casc, const uint8_t *d_gray, int W, int H, int gstride,
                     const uint8_t *d_lut, const nv_detect_params *p)
{
    int rc = detect_prepare(ctx, casc, W, H, p);
    if (rc != NV_OK) return rc;
    // A plan that sees the same (image, cascade, parameters) again replays its launches as one CUDA graph: the nested
    // ROI stages of the eye / mouth / nose / ear elements call this several times per frame on tiny images, where the
    // launches cost more than the kernels.  Debug / profiling runs keep individual launches (taps and events).
    PlanSlot *sl = ctx->ps;
    DetGraphKey key;
    key.gray = d_gray; key.gstride = gstride; key.lut = d_lut; key.casc = casc->uid; key.sf = p->scale_factor; key.mn = p->min_neighbors;
    key.epoch = ctx->epoch; key.scores = ctx->scores;
    bool graphable = !ctx->debug && !ctx->profile && !ctx->no_graph;
    int nl = 0;
    if (graphable && sl->dexec && key == sl->dkey) {
        NV_CUDA(cudaGraphLaunch(sl->dexec, ctx->stream));
        nl = sl->d_nl;
    } else if (graphable && key == sl->dkey_seen) {
        if (sl->dexec) { cudaGraphExecDestroy(sl->dexec); sl->dexec = nullptr; }
        cudaGraph_t g = nullptr;
        NV_CUDA(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
        rc = detect_enqueue(ctx, casc, d_gray, W, H, gstride, d_lut, p, &nl);
        cudaError_t ce = cudaStreamEndCapture(ctx->stream, &g);
        if (rc != NV_OK || ce != cudaSuccess || !g) {
            if (g) cudaGraphDestroy(g);
            cudaGetLastError();
            ctx->no_graph = true;                      // capture is not possible here: stay on plain launches
            nl = 0;
            if ((rc = detect_enqueue(ctx, casc, d_gray, W, H, gstride, d_lut, p, &nl)) != NV_OK) return rc;
        } else {
            ce = cudaGraphInstantiate(&sl->dexec, g, 0);
            cudaGraphDestroy(g);
            if (ce != cudaSuccess) { sl->dexec = nullptr; nv_set_error("cudaGraphInstantiate: %s", cudaGetErrorString(ce)); return NV_ERR_CUDA; }
            sl->dkey = key; sl->d_nl = nl;
            NV_CUDA(cudaGraphLaunch(sl->dexec, ctx->stream));
        }
    } else {
        sl->dkey_seen = key;
        if ((rc = detect_enqueue(ctx, casc, d_gray, W, H, gstride, d_lut, p, &nl)) != NV_OK) return rc;
    }
    ctx->launches += nl;
    detect_bookkeeping(ctx, casc, d_gray, W, H, gstride, d_lut, p);
    return NV_OK;
}

int nv_collect(nv_ctx *ctx, nv_rect *out, int cap, int *n)
{
    if (!ctx->pending) { nv_set_error("collect without a pending submit"); return NV_ERR_STATE; }
    NV_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->pending = false;
    const ResultHeader *h = reinterpret_cast<const ResultHeader *>(ctx->h_result);
    if (h->overflow) {
        // raw candidates outgrew the buffers: grow them and run the same call again (inputs are still on the device)
        int need = h->n_cand, lim = ctx->last_min_neighbors > 0 ? CAND_CAP_GROUPED : CAND_CAP_RAW;
        if (need > lim || need <= ctx->cand_cap) {
            nv_set_error("%d raw candidates exceed the supported maximum of %d", need, lim);
            return NV_ERR_CAPACITY;
        }
        int rc = alloc_candidates(ctx, std::min(lim, need + need / 4 + 64), ctx->last_min_neighbors > 0);
        if (rc != NV_OK) return rc;
        nv_detect_params p = ctx->last_params;
        const int scores = ctx->scores;
        ctx->scores = ctx->last_scores;                      // the call as it was submitted
        rc = nv_detect_device(ctx, ctx->last_casc, ctx->tap_gray, ctx->last_W, ctx->last_H, ctx->tap_stride, ctx->tap_lut, &p);
        ctx->scores = scores;
        if (rc != NV_OK) return rc;
        NV_CUDA(cudaStreamSynchronize(ctx->stream));
        ctx->pending = false;
        h = reinterpret_cast<const ResultHeader *>(ctx->h_result);
    }
    int total = h->n_out;
    if (total > NV_RESULT_INLINE) {
        NV_CUDA(cudaMemcpy(ctx->h_result + sizeof(ResultHeader) + NV_RESULT_INLINE * sizeof(nv_rect),
                           ctx->d_result + sizeof(ResultHeader) + NV_RESULT_INLINE * sizeof(nv_rect),
                           (size_t)(total - NV_RESULT_INLINE) * sizeof(nv_rect), cudaMemcpyDeviceToHost));
        if (ctx->last_scores) {
            const size_t wofs = sizeof(ResultHeader) + (size_t)ctx->result_cap * sizeof(nv_rect), nofs = wofs + (size_t)ctx->result_cap * sizeof(double);
            NV_CUDA(cudaMemcpy(ctx->h_result + wofs + NV_RESULT_INLINE * sizeof(double), ctx->d_result + wofs + NV_RESULT_INLINE * sizeof(double),
                               (size_t)(total - NV_RESULT_INLINE) * sizeof(double), cudaMemcpyDeviceToHost));
            NV_CUDA(cudaMemcpy(ctx->h_result + nofs + NV_RESULT_INLINE * sizeof(int), ctx->d_result + nofs + NV_RESULT_INLINE * sizeof(int),
                               (size_t)(total - NV_RESULT_INLINE) * sizeof(int), cudaMemcpyDeviceToHost));
        }
    }
    ctx->scores_ready = ctx->last_scores;
    int m = std::min(total, cap);
    if (out && m > 0) memcpy(out, ctx->h_result + sizeof(ResultHeader), (size_t)m * sizeof(nv_rect));
    if (n) *n = m;
    if (h->overflow) {
        nv_set_error("internal capacity exceeded (%d raw candidates, cap %d)", h->n_cand, ctx->cand_cap);
        return NV_ERR_CAPACITY;
    }
    if (total > cap) { nv_set_error("%d rectangles, caller capacity %d", total, cap); return NV_ERR_CAPACITY; }
    return NV_OK;
}

// host -> device copy of an input image on the ctx's stream: page-locked caller memory is read directly by the
// DMA engine, pageable memory goes through the ctx's pinned staging buffer
int nv_h2d(nv_ctx *ctx, const uint8_t *src, size_t bytes)
{
    cudaPointerAttributes at;
    bool known = cudaPointerGetAttributes(&at, src) == cudaSuccess;
    if (known && (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged)) {
        // a frame that already lives in device memory (nv_element_transform_frame_device): one copy inside HBM
        NV_CUDA(cudaMemcpyAsync(ctx->d_frame, src, bytes, cudaMemcpyDeviceToDevice, ctx->stream));
        return NV_OK;
    }
    bool pinned = known && at.type == cudaMemoryTypeHost;
    if (!pinned) { cudaGetLastError(); memcpy(ctx->h_frame, src, bytes); }
    NV_CUDA(cudaMemcpyAsync(ctx->d_frame, pinned ? src : ctx->h_frame, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return NV_OK;
}

static int check_frame(nv_ctx *ctx, const void *img, int w, int h, int stride, int cn)
{
    if (!ctx || !img) { nv_set_error("null argument"); return NV_ERR_ARG; }
    if (w <= 0 || h <= 0 || stride < w * cn) { nv_set_error("bad frame geometry %dx%d stride %d", w, h, stride); return NV_ERR_ARG; }
    if (w > ctx->max_w || h > ctx->max_h || (size_t)stride * h > ctx->frame_cap) {
        nv_set_error("frame %dx%d exceeds the context's %dx%d", w, h, ctx->max_w, ctx->max_h);
        return NV_ERR_CAPACITY;
    }
    return NV_OK;
}

extern "C" int nv_detect_multiscale(nv_ctx *ctx, const nv_cascade *c, const uint8_t *gray, int width, int height,
                                    int stride_bytes, const nv_detect_params *p, nv_rect *out, int cap, int *n)
{
    int rc = check_frame(ctx, gray, width, height, stride_bytes, 1);
    if (rc != NV_OK) return rc;
    if (!c || !p) { nv_set_error("null argument"); return NV_ERR_ARG; }
    NV_CUDA(cudaSetDevice(ctx->gpu));
    if (ctx->pending) NV_CUDA(cudaStreamSynchronize(ctx->stream));
    if ((rc = nv_h2d(ctx, gray, (size_t)stride_bytes * height)) != NV_OK) return rc;
    rc = nv_detect_device(ctx, const_cast<nv_cascade *>(c), ctx->d_frame, width, height, stride_bytes, ctx->d_lut + 256, p);
    if (rc != NV_OK) return rc;
    return nv_collect(ctx, out, cap, n);
}

// ------------------------------------------------------------------------------------------------
// face element hot block
// ------------------------------------------------------------------------------------------------
int nv_get_rtab(nv_ctx *ctx, int sw, int sh, int dw, int dh, const int **d_tab, const nv_ctx::RtabEntry **entry)
{
    ResizeKey k;
    k.sw = sw; k.sh = sh; k.dw = dw; k.dh = dh;
    for (auto &e : ctx->rtabs)
        if (e.d && e.k == k) { *d_tab = e.d; if (entry) *entry = &e; return NV_OK; }
    std::vector<int> tab;
    build_resize_tables(sw, sh, dw, dh, tab);
    nv_ctx::RtabEntry &e = ctx->rtabs[ctx->rtab_next];
    ctx->rtab_next = (ctx->rtab_next + 1) % 16;
    if (e.d) {
        NV_CUDA(cudaStreamSynchronize(ctx->stream));       // an in-flight kernel may still read the evicted table
        NV_CUDA(cudaFree(e.d));
        e.d = nullptr;
    }
    NV_CUDA(cudaMalloc(&e.d, tab.size() * sizeof(int)));
    NV_CUDA(cudaMemcpyAsync(e.d, tab.data(), tab.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    NV_CUDA(cudaStreamSynchronize(ctx->stream));           // tab is a local
    e.k = k;
    e.row_a = e.row_period = 0;
    if (tab[0] == RT_LINEAR && dh >= 2) {                  // which source rows does the vertical pass read?
        const int *y0 = &tab[1 + 2 * (size_t)dw], *y1 = y0 + dh;
        const int per = y0[1] - y0[0];
        bool regular = per >= 3;
        for (int dy = 0; dy < dh && regular; dy++) regular = y0[dy] == y0[0] + per * dy && y1[dy] == y0[dy] + 1;
        if (regular) { e.row_a = y0[0]; e.row_period = per; }
    }
    *d_tab = e.d;
    if (entry) *entry = &e;
    return NV_OK;
}

// Host frame -> ctx->d_frame, only the row pairs an integer down-scale reads (RtabEntry::row_period): `n` pairs of rows
// a + k * period, a + k * period + 1, at their own offsets, as one strided copy — half the bytes of a 640x480 frame that
// is processed at 160x120.  Page-locked caller memory is read in place, anything else goes through the staging buffer.
static int nv_h2d_row_pairs(nv_ctx *ctx, const uint8_t *src, int stride, int height, int a, int period, int n)
{
    cudaPointerAttributes at;
    bool known = cudaPointerGetAttributes(&at, src) == cudaSuccess;
    if (known && (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged)) return nv_h2d(ctx, src, (size_t)stride * height);
    const bool pinned = known && at.type == cudaMemoryTypeHost;
    const size_t off = (size_t)a * stride, pitch = (size_t)period * stride, run = 2 * (size_t)stride;
    if (!pinned) {
        cudaGetLastError();
        for (int k = 0; k < n; k++) memcpy(ctx->h_frame + off + k * pitch, src + off + k * pitch, run);
    }
    NV_CUDA(cudaMemcpy2DAsync(ctx->d_frame + off, pitch, (pinned ? src : ctx->h_frame) + off, pitch, run, n, cudaMemcpyHostToDevice, ctx->stream));
    return NV_OK;
}

// Source frame of the face block: interleaved BGR (p[0], s[0]) or the planes of a 4:2:0 frame.
struct FaceSrc { int fmt; const uint8_t *p[3]; int s[3]; bool on_device; };

// Host planes of a 4:2:0 frame -> ctx->d_frame.  Planes that lie in one ascending block of host memory (a GstVideoFrame
// mapped from a single GstMemory, a cv::Mat of h*3/2 rows) travel as ONE copy and keep their relative offsets; scattered
// planes are copied one by one to 256-byte aligned offsets.  Fills the device plane pointers.
static int yuv_h2d(nv_ctx *ctx, const FaceSrc &f, int height, SrcPlanes *d)
{
    int np = f.fmt == NV_FMT_I420 ? 3 : 2;
    size_t bytes[3] = {(size_t)f.s[0] * height, (size_t)f.s[1] * (height / 2), np == 3 ? (size_t)f.s[2] * (height / 2) : 0};
    // tight end of the last row of a plane does not matter: strides are honoured, the tail padding is copied along
    // Only planes that follow each other with at most a row (or 256 bytes) of padding between them are taken as one block:
    // a larger gap means separate allocations that merely happen to ascend, and the bytes between them are not the caller's.
    const uint8_t *lo = f.p[0], *hi = f.p[0] + bytes[0];
    bool block = true;
    for (int i = 1; i < np; i++) {
        const size_t max_gap = std::max<size_t>(256, (size_t)f.s[i - 1]);
        if (f.p[i] < hi || (size_t)(f.p[i] - hi) > max_gap || (size_t)(f.p[i] - lo) + bytes[i] > ctx->frame_cap) { block = false; break; }
        hi = f.p[i] + bytes[i];
    }
    size_t off[3] = {0, 0, 0};
    if (block) {
        for (int i = 1; i < np; i++) off[i] = (size_t)(f.p[i] - lo);
        int rc = nv_h2d(ctx, lo, (size_t)(hi - lo));
        if (rc != NV_OK) return rc;
    } else {
        size_t o = 0;
        for (int i = 0; i < np; i++) { off[i] = o; o += (bytes[i] + 255) & ~(size_t)255; }
        if (o > ctx->frame_cap) { nv_set_error("4:2:0 frame larger than the context"); return NV_ERR_CAPACITY; }
        for (int i = 0; i < np; i++) {
            cudaPointerAttributes at;
            bool pinned = cudaPointerGetAttributes(&at, f.p[i]) == cudaSuccess && at.type == cudaMemoryTypeHost;
            if (!pinned) { cudaGetLastError(); memcpy(ctx->h_frame + off[i], f.p[i], bytes[i]); }
            NV_CUDA(cudaMemcpyAsync(ctx->d_frame + off[i], pinned ? f.p[i] : ctx->h_frame + off[i], bytes[i],
                                    cudaMemcpyHostToDevice, ctx->stream));
        }
    }
    d->p0 = ctx->d_frame; d->p1 = ctx->d_frame + off[1]; d->p2 = np == 3 ? ctx->d_frame + off[2] : nullptr;
    d->s0 = f.s[0]; d->s1 = f.s[1]; d->s2 = f.s[2];
    return NV_OK;
}

static int check_yuv(nv_ctx *ctx, const nv_yuv_frame *f, FaceSrc *src)
{
    if (!ctx || !f || !f->plane[0] || !f->plane[1]) { nv_set_error("null argument"); return NV_ERR_ARG; }
    if (f->format != NV_FMT_I420 && f->format != NV_FMT_NV12 && f->format != NV_FMT_NV21) {
        nv_set_error("format %d is not a 4:2:0 nv_pixel_format", f->format); return NV_ERR_ARG;
    }
    bool planar = f->format == NV_FMT_I420;
    int w = f->width, h = f->height;
    if (w <= 0 || h <= 0 || (w & 1) || (h & 1)) { nv_set_error("4:2:0 frame needs even, positive width and height (%dx%d)", w, h); return NV_ERR_ARG; }
    if (f->stride[0] < w || f->stride[1] < (planar ? w / 2 : w) || (planar && (!f->plane[2] || f->stride[2] < w / 2))) {
        nv_set_error("bad 4:2:0 plane geometry"); return NV_ERR_ARG;
    }
    size_t total = (size_t)f->stride[0] * h + (size_t)f->stride[1] * (h / 2) + (planar ? (size_t)f->stride[2] * (h / 2) : 0);
    if (w > ctx->max_w || h > ctx->max_h || total + 768 > ctx->frame_cap) {
        nv_set_error("frame %dx%d exceeds the context's %dx%d", w, h, ctx->max_w, ctx->max_h); return NV_ERR_CAPACITY;
    }
    src->fmt = f->format; src->on_device = f->on_device != 0;
    for (int i = 0; i < 3; i++) { src->p[i] = f->plane[i]; src->s[i] = f->stride[i]; }
    if (!planar) { src->p[2] = nullptr; src->s[2] = 0; }
    return NV_OK;
}

int nv_yuv_upload(nv_ctx *ctx, const nv_yuv_frame *f, SrcPlanes *planes)
{
    FaceSrc src;
    int rc = check_yuv(ctx, f, &src);
    if (rc != NV_OK) return rc;
    NV_CUDA(cudaSetDevice(ctx->gpu));
    if (ctx->pending) NV_CUDA(cudaStreamSynchronize(ctx->stream));
    *planes = SrcPlanes{src.p[0], src.p[1], src.p[2], src.s[0], src.s[1], src.s[2]};
    return src.on_device ? NV_OK : yuv_h2d(ctx, src, f->height, planes);
}

// The face element's processing size and detect parameters (kmsfacedetect.cpp:304, integer division, :770-777, :811).
static void face_geometry(int width, int height, const nv_face_params *p, int *cols, int *rows, nv_detect_params *dp)
{
    int iscale = width / p->width_to_process;
    double scale = iscale;
    *rows = height; *cols = width;
    if (iscale > 0 && cv_round(height / scale) > 0) *rows = cv_round(height / scale); else scale = 1;
    if (scale > 0 && cv_round(width / scale) > 0) *cols = cv_round(width / scale); else scale = 1;
    dp->scale_factor = p->scale_factor; dp->min_neighbors = p->min_neighbors; dp->flags = 0;
    dp->min_w = p->min_w < 0 ? *cols / 20 : p->min_w;
    dp->min_h = p->min_w < 0 ? *rows / 20 : p->min_h;
    dp->max_w = dp->max_h = 0;
}

static int face_submit_impl(nv_ctx *ctx, const nv_cascade *c, const FaceSrc &src, int width, int height, const nv_face_params *p)
{
    const uint8_t *bgr = src.p[0];
    const bool on_device = src.on_device, yuv = src.fmt != NV_FMT_BGR;
    const int stride = src.s[0];
    if (!ctx || !c || !bgr || !p) { nv_set_error("null argument"); return NV_ERR_ARG; }
    if (p->width_to_process <= 0) { nv_set_error("width_to_process must be > 0 (kmsfacedetect.cpp:304 divides by it)"); return NV_ERR_ARG; }
    int rc;
    if (yuv) { /* geometry checked by check_yuv */ }
    else if (!on_device) { if ((rc = check_frame(ctx, bgr, width, height, stride, 3)) != NV_OK) return rc; }
    else if (width <= 0 || height <= 0 || width > ctx->max_w || height > ctx->max_h || stride < 3 * width) {
        nv_set_error("bad device frame geometry"); return NV_ERR_ARG;
    }
    NV_CUDA(cudaSetDevice(ctx->gpu));
    if (ctx->pending) NV_CUDA(cudaStreamSynchronize(ctx->stream));
    int rows, cols;
    nv_detect_params dp;
    face_geometry(width, height, p, &cols, &rows, &dp);
    const int *d_rtab;
    const nv_ctx::RtabEntry *rt = nullptr;
    if ((rc = nv_get_rtab(ctx, width, height, cols, rows, &d_rtab, &rt)) != NV_OK) return rc;
    const int row_a = rt->row_a, row_period = rt->row_period;         // (the entry may be evicted by a later call)
    nv_cascade *casc = const_cast<nv_cascade *>(c);
    if ((rc = detect_prepare(ctx, casc, cols, rows, &dp)) != NV_OK) return rc;

    const uint8_t *d_src = bgr;
    SrcPlanes planes = {src.p[0], src.p[1], src.p[2], src.s[0], src.s[1], src.s[2]};
    if (!on_device) {
        // page-locked caller memory is copied straight from the caller; anything else goes through the pinned staging buffer
        if (yuv) { if ((rc = yuv_h2d(ctx, src, height, &planes)) != NV_OK) return rc; }
        else if (row_period > 0) { if ((rc = nv_h2d_row_pairs(ctx, bgr, stride, height, row_a, row_period, rows)) != NV_OK) return rc; }
        else if ((rc = nv_h2d(ctx, bgr, (size_t)stride * height)) != NV_OK) return rc;
        d_src = ctx->d_frame;
    }
    auto enqueue = [&](int *nl) -> int {
        ctx->prof_set[0] = ctx->prof_set[1] = false;
        prof_mark(ctx, 0);
        // the prep kernel's last block turns the histogram into the equalizeHist LUT (no launch of its own for the LUT; the "hist_lut" stage of
        // the profile is empty)
        if (yuv) NV_CUDA(launch_face_prep_yuv(src.fmt, planes, width, height, ctx->d_gray, cols, rows, d_rtab, ctx->d_hist, ctx->stream, ctx->d_lut));
        else NV_CUDA(launch_face_prep(d_src, width, height, stride, 3, ctx->d_gray, cols, rows, d_rtab, ctx->d_hist, ctx->stream, ctx->d_lut));
        prof_mark(ctx, 1);
        *nl += 1;
        return detect_enqueue(ctx, casc, ctx->d_gray, cols, rows, cols, ctx->d_lut, &dp, nl);
    };
    // A context that sees the same call shape again replays it as ONE CUDA graph launch (the per-stream steady
    // state of an element); debug / profiling runs keep individual launches so that their events and taps work.
    nv_ctx::GraphKey key = {d_src, width, height, stride, cols, rows, d_rtab, casc->uid, dp.scale_factor, dp.min_neighbors,
                            dp.min_w, dp.min_h, ctx->epoch, ctx->ps, ctx->ps->gen,
                            src.fmt, yuv ? planes.p1 : nullptr, yuv ? planes.p2 : nullptr, yuv ? planes.s1 : 0, yuv ? planes.s2 : 0,
                            ctx->scores};
    bool graphable = !ctx->debug && !ctx->no_graph;
    int nl = 0;
    if (graphable && ctx->gexec && key == ctx->gkey) {
        NV_CUDA(cudaGraphLaunch(ctx->gexec, ctx->stream));
        nl = ctx->g_nl;
        for (int i = 0; i <= NV_NUM_STAGES; i++) ctx->prof_set[i] = ctx->profile && ((ctx->g_prof_mask >> i) & 1u);
    } else if (graphable && key == ctx->gkey_seen) {
        if (ctx->gexec) { cudaGraphExecDestroy(ctx->gexec); ctx->gexec = nullptr; }
        cudaGraph_t g = nullptr;
        NV_CUDA(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
        rc = enqueue(&nl);
        cudaError_t ce = cudaStreamEndCapture(ctx->stream, &g);
        if (rc != NV_OK || ce != cudaSuccess || !g) {
            if (g) cudaGraphDestroy(g);
            cudaGetLastError();
            ctx->no_graph = true;                      // capture is not possible here: stay on plain launches
            nl = 0;
            if ((rc = enqueue(&nl)) != NV_OK) return rc;
        } else {
            ce = cudaGraphInstantiate(&ctx->gexec, g, 0);
            cudaGraphDestroy(g);
            if (ce != cudaSuccess) { ctx->gexec = nullptr; nv_set_error("cudaGraphInstantiate: %s", cudaGetErrorString(ce)); return NV_ERR_CUDA; }
            ctx->gkey = key; ctx->g_nl = nl;
            ctx->g_prof_mask = 0;
            for (int i = 0; i <= NV_NUM_STAGES; i++) if (ctx->prof_set[i]) ctx->g_prof_mask |= 1u << i;
            NV_CUDA(cudaGraphLaunch(ctx->gexec, ctx->stream));
        }
    } else {
        ctx->gkey_seen = key;
        if ((rc = enqueue(&nl)) != NV_OK) return rc;
    }
    ctx->launches += nl;
    detect_bookkeeping(ctx, casc, ctx->d_gray, cols, rows, cols, ctx->d_lut, &dp);
    return NV_OK;
}

extern "C" int nv_face_submit(nv_ctx *ctx, const nv_cascade *c, const uint8_t *bgr, int width, int height,
                              int stride_bytes, const nv_face_params *p)
{
    FaceSrc src = {NV_FMT_BGR, {bgr, nullptr, nullptr}, {stride_bytes, 0, 0}, false};
    return face_submit_impl(ctx, c, src, width, height, p);
}

extern "C" int nv_face_submit_device(nv_ctx *ctx, const nv_cascade *c, const uint8_t *d_bgr, int width, int height,
                                     int stride_bytes, const nv_face_params *p)
{
    FaceSrc src = {NV_FMT_BGR, {d_bgr, nullptr, nullptr}, {stride_bytes, 0, 0}, true};
    return face_submit_impl(ctx, c, src, width, height, p);
}

extern "C" int nv_host_alloc(size_t bytes, void **out)
{
    if (!out || !bytes) { nv_set_error("null argument"); return NV_ERR_ARG; }
    if (nv_device_count() < 1) { nv_set_error("no CUDA device"); return NV_ERR_NO_DEVICE; }
    NV_CUDA(cudaHostAlloc(out, bytes, cudaHostAllocPortable));
    return NV_OK;
}

extern "C" void nv_host_free(void *p) { if (p) cudaFreeHost(p); }

// Page-lock memory the caller already owns (a block of the upstream buffer pool): frames inside it are then read by the
// DMA engine directly, without the staging copy a pageable frame costs.
extern "C" int nv_host_register(void *p, size_t bytes)
{
    if (!p || !bytes) { nv_set_error("null argument"); return NV_ERR_ARG; }
    if (nv_device_count() < 1) { nv_set_error("no CUDA device"); return NV_ERR_NO_DEVICE; }
    NV_CUDA(cudaHostRegister(p, bytes, cudaHostRegisterPortable));
    return NV_OK;
}

extern "C" int nv_host_unregister(void *p)
{
    if (!p) { nv_set_error("null argument"); return NV_ERR_ARG; }
    NV_CUDA(cudaHostUnregister(p));
    return NV_OK;
}

extern "C" int nv_face_submit_yuv(nv_ctx *ctx, const nv_cascade *c, const nv_yuv_frame *f, const nv_face_params *p)
{
    FaceSrc src;
    int rc = check_yuv(ctx, f, &src);
    if (rc != NV_OK) return rc;
    return face_submit_impl(ctx, c, src, f->width, f->height, p);
}

extern "C" int nv_face_detect_yuv(nv_ctx *ctx, const nv_cascade *c, const nv_yuv_frame *f, const nv_face_params *p,
                                  nv_rect *out, int cap, int *n)
{
    int rc = nv_face_submit_yuv(ctx, c, f, p);
    if (rc != NV_OK) return rc;
    return nv_face_collect(ctx, out, cap, n);
}

extern "C" int nv_face_collect(nv_ctx *ctx, nv_rect *out, int cap, int *n)
{
    if (!ctx) { nv_set_error("null ctx"); return NV_ERR_ARG; }
    if (ctx->batch_last) { nv_set_error("the pending call is a batch: collect it with nv_face_collect_batch"); return NV_ERR_STATE; }
    NV_CUDA(cudaSetDevice(ctx->gpu));
    return nv_collect(ctx, out, cap, n);
}

extern "C" int nv_face_detect(nv_ctx *ctx, const nv_cascade *c, const uint8_t *bgr, int width, int height,
                              int stride_bytes, const nv_face_params *p, nv_rect *out, int cap, int *n)
{
    int rc = nv_face_submit(ctx, c, bgr, width, height, stride_bytes, p);
    if (rc != NV_OK) return rc;
    return nv_face_collect(ctx, out, cap, n);
}

// ------------------------------------------------------------------------------------------------
// batches: N same-size images per call
// ------------------------------------------------------------------------------------------------
// The batched route runs the small-plan chain of a cascade with the exactness certificates (k_stage0_rows_p, k_cascade_tail_tab
// over all stages, k_group_fused) once for the whole batch: every kernel takes the image as a grid dimension, all images share
// the plan, and the alive windows of all images share one queue.  Anything else runs the single-image pipeline once per image.
static bool batch_routable(const nv_ctx *ctx, const nv_cascade *casc)
{
    const PlanDev &P = ctx->ps->plan;
    return P.nlevels > 0 && P.total_windows <= NV_SMALL_PLAN_WINDOWS && !casc->h.general && casc->tail_fast && ctx->cur_tail &&
           ctx->ps->use_s0p && casc->meta.nstages > 1 && tail_tab_smem(casc->meta, 1, casc->meta.nstages) <= NV_TAILTAB_MAX_SMEM;
}

static void batch_free(nv_ctx::Batch &b)
{
    cudaFree(b.d_frame); cudaFreeHost(b.h_stage); cudaFree(b.d_gray); cudaFree(b.d_lut); cudaFree(b.d_hist); cudaFree(b.d_sum);
    cudaFree(b.d_sq); cudaFree(b.d_bits); cudaFree(b.d_vnf); cudaFree(b.d_queue); cudaFree(b.d_cand); cudaFree(b.d_sorted);
    cudaFree(b.d_rects); cudaFree(b.d_adj); cudaFree(b.d_grp); cudaFree(b.d_counters); cudaFree(b.d_result); cudaFreeHost(b.h_result);
    cudaFree(b.d_tab); cudaFreeHost(b.h_tab);
    const unsigned long long gen = b.gen;
    b = nv_ctx::Batch();
    b.gen = gen + 1;
}

#define BATCH_RESULT_BYTES (sizeof(ResultHeader) + (size_t)NV_BATCH_GROUP_CAP * sizeof(nv_rect))
#define BATCH_ADJ_WORDS ((size_t)NV_BATCH_GROUP_CAP * (NV_BATCH_GROUP_CAP / 32))

// per-image buffers of the batched route for n images of this plan (grow-only); staging only when a pageable frame needs it
static int batch_buffers(nv_ctx *ctx, int n, size_t frame_bytes, size_t gray_bytes, bool stage)
{
    nv_ctx::Batch &b = ctx->b;
    const PlanDev &P = ctx->ps->plan;
    const LevelDesc &Lz = P.lv[P.nlevels - 1];
    const size_t integ = align_up((int)((size_t)Lz.iofs + (size_t)Lz.ipitch * (Lz.lh + 1)), 64);
    const size_t wins = align_up(P.total_windows, 64), bits = align_up(Lz.bofs + Lz.nxw * Lz.ny, 64);
    if (n > b.cap || frame_bytes > b.frame_bytes || gray_bytes > b.gray_bytes || integ > b.integ || wins > b.wins || bits > b.bits) {
        NV_CUDA(cudaStreamSynchronize(ctx->stream));
        const bool had_stage = b.h_stage != nullptr;
        const nv_ctx::Batch old = b;
        batch_free(b);
        b.cap = std::max(n, old.cap); b.frame_bytes = std::max(frame_bytes, old.frame_bytes); b.gray_bytes = std::max(gray_bytes, old.gray_bytes);
        b.integ = std::max(integ, old.integ); b.wins = std::max(wins, old.wins); b.bits = std::max(bits, old.bits);
        // sizes are committed above; should any allocation fail, everything is released again (capacity 0), so that
        // the next call allocates afresh instead of running on missing buffers
        const int rc = [&]() -> int {
            const size_t N = (size_t)b.cap, G = NV_BATCH_GROUP_CAP;
            NV_CUDA(cudaMalloc(&b.d_frame, N * b.frame_bytes));
            if (had_stage) NV_CUDA(cudaMallocHost(&b.h_stage, N * b.frame_bytes));
            NV_CUDA(cudaMalloc(&b.d_gray, N * b.gray_bytes));
            NV_CUDA(cudaMalloc(&b.d_lut, N * 256));
            NV_CUDA(cudaMalloc(&b.d_hist, N * NV_HIST_STRIDE * sizeof(int)));
            NV_CUDA(cudaMemset(b.d_hist, 0, N * NV_HIST_STRIDE * sizeof(int)));       // the prep kernel's last block leaves it zeroed
            NV_CUDA(cudaMalloc(&b.d_sum, N * b.integ * sizeof(uint32_t)));
            NV_CUDA(cudaMemset(b.d_sum, 0, N * b.integ * sizeof(uint32_t)));
            NV_CUDA(cudaMalloc(&b.d_sq, N * b.integ * sizeof(uint32_t)));
            NV_CUDA(cudaMemset(b.d_sq, 0, N * b.integ * sizeof(uint32_t)));
            NV_CUDA(cudaMalloc(&b.d_bits, N * b.bits * sizeof(uint32_t)));
            NV_CUDA(cudaMalloc(&b.d_vnf, N * b.wins * sizeof(float)));
            NV_CUDA(cudaMalloc(&b.d_queue, N * b.wins * sizeof(uint2)));
            NV_CUDA(cudaMalloc(&b.d_cand, N * b.wins * sizeof(uint32_t)));
            NV_CUDA(cudaMalloc(&b.d_sorted, N * G * sizeof(uint32_t)));
            NV_CUDA(cudaMalloc(&b.d_rects, N * G * sizeof(int4)));
            NV_CUDA(cudaMalloc(&b.d_adj, N * BATCH_ADJ_WORDS * sizeof(uint32_t)));
            NV_CUDA(cudaMalloc(&b.d_grp, N * 8 * G * sizeof(int)));
            NV_CUDA(cudaMalloc(&b.d_counters, 16 * (N + 1) * sizeof(int)));
            NV_CUDA(cudaMemset(b.d_counters, 0, 16 * (N + 1) * sizeof(int)));      // from here on k_group_fused leaves them at zero
            NV_CUDA(cudaMalloc(&b.d_result, N * BATCH_RESULT_BYTES));
            NV_CUDA(cudaMallocHost(&b.h_result, N * BATCH_RESULT_BYTES));
            memset(b.h_result, 0, N * BATCH_RESULT_BYTES);
            NV_CUDA(cudaMalloc(&b.d_tab, 2 * N * sizeof(uint8_t *)));
            NV_CUDA(cudaMallocHost(&b.h_tab, 2 * N * sizeof(uint8_t *)));
            return NV_OK;
        }();
        if (rc != NV_OK) { batch_free(b); return rc; }
    }
    if (stage && !b.h_stage) NV_CUDA(cudaMallocHost(&b.h_stage, (size_t)b.cap * b.frame_bytes));
    return NV_OK;
}

// host frame -> device: whole frame (period == 0) or the row pairs a + k * period, + 1 that an integer down-scale reads.
// Page-locked memory (type cudaMemoryTypeHost) is read in place, pageable memory goes through `stage`, device memory is
// copied inside HBM.
static int batch_upload(nv_ctx *ctx, uint8_t *dst, uint8_t *stage, const uint8_t *src, cudaMemoryType type, int stride, int height, int a,
                        int period, int n)
{
    if (type == cudaMemoryTypeDevice || type == cudaMemoryTypeManaged) {
        NV_CUDA(cudaMemcpyAsync(dst, src, (size_t)stride * height, cudaMemcpyDeviceToDevice, ctx->stream));
        return NV_OK;
    }
    const bool pinned = type == cudaMemoryTypeHost;
    if (period <= 0) {
        if (!pinned) memcpy(stage, src, (size_t)stride * height);
        NV_CUDA(cudaMemcpyAsync(dst, pinned ? src : stage, (size_t)stride * height, cudaMemcpyHostToDevice, ctx->stream));
        return NV_OK;
    }
    const size_t off = (size_t)a * stride, pitch = (size_t)period * stride, run = 2 * (size_t)stride;
    if (!pinned)
        for (int k = 0; k < n; k++) memcpy(stage + off + k * pitch, src + off + k * pitch, run);
    NV_CUDA(cudaMemcpy2DAsync(dst + off, pitch, (pinned ? src : stage) + off, pitch, run, n, cudaMemcpyHostToDevice, ctx->stream));
    return NV_OK;
}

enum { BATCH_GRAY = 1, BATCH_FACE = 2 };

// the stream-ordered chain of the batched route: six launches whatever n is (five for gray images)
static int batch_enqueue(nv_ctx *ctx, nv_cascade *casc, int kind, int n, int w, int h, int stride, int cols, int rows, const int *rtab,
                         bool aligned, int min_neighbors, int *nlaunch)
{
    nv_ctx::Batch &b = ctx->b;
    const PlanDev &P = ctx->ps->plan;
    cudaStream_t st = ctx->stream;
    const int qcap = (int)(n * b.wins);
    const uint8_t *const *grays = b.d_tab;
    const uint8_t *lut = ctx->d_lut + 256;                   // gray images: the identity LUT
    int lut_stride = 0, gstride = stride, nl = 0;
    if (kind == BATCH_FACE) {
        NV_CUDA(launch_face_prep_batch(b.d_tab, n, aligned, w, h, stride, b.d_gray, cols, rows, rtab, b.d_hist, b.d_lut, st));
        grays = b.d_tab + n; lut = b.d_lut; lut_stride = 256; gstride = cols; nl++;
    }
    NV_CUDA(launch_pyramid_batch(ctx->ps->d_plan, P.total_rowblk, P.total_colblk, n, grays, gstride, lut, lut_stride, ctx->ps->d_ptab,
                                 b.d_sum, b.d_sq, b.integ, st));
    Stage0Params &sp = ctx->ps->s0p;
    sp.sum = b.d_sum; sp.sq = b.d_sq; sp.vnf = b.d_vnf; sp.bits_alive = b.d_bits; sp.counters = b.d_counters; sp.depth = nullptr;
    sp.queue = b.d_queue; sp.queue_cap = qcap; sp.queue_cidx = 3;
    sp.integ_stride = b.integ; sp.win_stride = (int)b.wins; sp.bits_stride = (int)b.bits;
    NV_CUDA(launch_stage0_rows_p_batch(sp, n, st));
    NV_CUDA(launch_cascade_tail_tab_batch(ctx->ps->d_plan, ctx->cur_meta, casc->meta, ctx->cur_tail, ctx->cur_tail_base, b.d_sum, b.integ,
                                          b.d_queue, qcap, b.d_counters, b.d_cand, (int)b.wins, st));
    NV_CUDA(launch_group_batch(ctx->ps->d_plan, n, b.d_counters, b.d_cand, (int)b.wins, NV_BATCH_GROUP_CAP, b.d_sorted, b.d_rects, b.d_adj,
                               BATCH_ADJ_WORDS, b.d_grp, min_neighbors, 0.2, cols, rows, b.d_result, b.h_result, BATCH_RESULT_BYTES, st));
    nl += 5;
    *nlaunch += nl;
    return NV_OK;
}

// one image of a batch through the single-image pipeline, collected into ctx->batch_out (appended; count in ctx->batch_counts[i])
static int batch_single(nv_ctx *ctx, int i, const uint8_t *src, bool on_device)
{
    int rc;
    if (ctx->batch_kind == BATCH_FACE) {
        FaceSrc fs = {NV_FMT_BGR, {src, nullptr, nullptr}, {ctx->batch_stride, 0, 0}, on_device};
        rc = face_submit_impl(ctx, ctx->batch_casc, fs, ctx->batch_w, ctx->batch_h, &ctx->batch_fp);
    } else {
        const uint8_t *d = src;
        if (!on_device) {
            if ((rc = nv_h2d(ctx, src, (size_t)ctx->batch_stride * ctx->batch_h)) != NV_OK) return rc;
            d = ctx->d_frame;
        }
        rc = nv_detect_device(ctx, ctx->batch_casc, d, ctx->batch_w, ctx->batch_h, ctx->batch_stride, ctx->d_lut + 256, &ctx->batch_dp);
    }
    if (rc != NV_OK) return rc;
    const size_t base = ctx->batch_out.size();
    ctx->batch_out.resize(base + CAND_CAP_RAW);
    int m = 0;
    rc = nv_collect(ctx, ctx->batch_out.data() + base, CAND_CAP_RAW, &m);
    ctx->batch_out.resize(base + (rc == NV_OK ? m : 0));
    if (rc != NV_OK) return rc;
    const ResultHeader *hd = reinterpret_cast<const ResultHeader *>(ctx->h_result);
    ctx->batch_counts[i] = m;
    ctx->batch_sum[0] += ctx->ps->plan.total_windows; ctx->batch_sum[1] += hd->n_alive; ctx->batch_sum[2] += hd->n_cand;
    return NV_OK;
}

static int batch_check(nv_ctx *ctx, const nv_cascade *c, const uint8_t *const *frames, int n, int w, int h, int stride, int cn,
                       const void *params)
{
    if (!ctx || !c || !frames || !params) { nv_set_error("null argument"); return NV_ERR_ARG; }
    if (n < 1 || n > NV_BATCH_MAX) { nv_set_error("batch of %d images: 1 .. %d are supported", n, NV_BATCH_MAX); return NV_ERR_ARG; }
    for (int i = 0; i < n; i++) if (!frames[i]) { nv_set_error("frame %d is null", i); return NV_ERR_ARG; }
    if (w <= 0 || h <= 0 || stride < w * cn) { nv_set_error("bad frame geometry %dx%d stride %d", w, h, stride); return NV_ERR_ARG; }
    if (w > ctx->max_w || h > ctx->max_h || (size_t)stride * h > ctx->frame_cap) {
        nv_set_error("frame %dx%d exceeds the context's %dx%d", w, h, ctx->max_w, ctx->max_h);
        return NV_ERR_CAPACITY;
    }
    if (ctx->scores) { nv_set_error("batch calls do not compute scores: switch them off with nv_ctx_set_scores(ctx, 0)"); return NV_ERR_STATE; }
    return NV_OK;
}

static int batch_submit(nv_ctx *ctx, nv_cascade *casc, int kind, const uint8_t *const *frames, int n, int w, int h, int stride,
                        bool on_device, const nv_face_params *fp, const nv_detect_params *gp)
{
    NV_CUDA(cudaSetDevice(ctx->gpu));
    if (ctx->pending) NV_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->pending = false;
    int rc, cols = w, rows = h, row_a = 0, row_period = 0;
    const int *d_rtab = nullptr;
    nv_detect_params dp;
    if (kind == BATCH_FACE) {
        if (fp->width_to_process <= 0) { nv_set_error("width_to_process must be > 0 (kmsfacedetect.cpp:304 divides by it)"); return NV_ERR_ARG; }
        face_geometry(w, h, fp, &cols, &rows, &dp);
        const nv_ctx::RtabEntry *rt = nullptr;
        if ((rc = nv_get_rtab(ctx, w, h, cols, rows, &d_rtab, &rt)) != NV_OK) return rc;
        row_a = rt->row_a; row_period = rt->row_period;
        ctx->batch_fp = *fp;
    } else {
        dp = *gp;
        ctx->batch_dp = *gp;
    }
    ctx->batch_casc = casc; ctx->batch_kind = kind; ctx->batch_n = n; ctx->batch_w = w; ctx->batch_h = h; ctx->batch_stride = stride;
    ctx->batch_on_device = on_device;
    ctx->batch_src.assign(frames, frames + n);
    ctx->batch_out.clear(); ctx->batch_counts.assign(n, 0);
    ctx->batch_sum[0] = ctx->batch_sum[1] = ctx->batch_sum[2] = 0;
    const long long launches0 = ctx->launches;
    if ((rc = detect_prepare(ctx, casc, cols, rows, &dp)) != NV_OK) return rc;
    ctx->batch_routed = batch_routable(ctx, casc);
    if (!ctx->batch_routed) {
        // sequential fallback: the single-image pipeline once per image, collected here
        for (int i = 0; i < n; i++)
            if ((rc = batch_single(ctx, i, frames[i], on_device)) != NV_OK) { ctx->batch_last = true; return rc; }
        ctx->batch_launches = ctx->launches - launches0;
        ctx->batch_last = true;
        ctx->pending = true;
        return NV_OK;
    }
    const size_t fbytes = (size_t)stride * h;
    bool pageable = false;
    std::vector<cudaMemoryType> types(on_device ? 0 : n);
    for (size_t i = 0; i < types.size(); i++) {
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, frames[i]) != cudaSuccess) { cudaGetLastError(); at.type = cudaMemoryTypeUnregistered; }
        types[i] = at.type;
        pageable = pageable || at.type == cudaMemoryTypeUnregistered;
    }
    if ((rc = batch_buffers(ctx, n, on_device ? 0 : fbytes, kind == BATCH_FACE ? (size_t)cols * rows : 0, pageable)) != NV_OK) return rc;
    nv_ctx::Batch &b = ctx->b;
    bool aligned = (stride & 3) == 0;
    for (int i = 0; i < n; i++) {
        const uint8_t *d = frames[i];
        if (!on_device) {
            uint8_t *dst = b.d_frame + i * fbytes;
            if ((rc = batch_upload(ctx, dst, b.h_stage ? b.h_stage + i * fbytes : nullptr, frames[i], types[i], stride, h,
                                   kind == BATCH_FACE ? row_a : 0, kind == BATCH_FACE ? row_period : 0, rows)) != NV_OK) return rc;
            d = dst;
        }
        aligned = aligned && ((uintptr_t)d & 3u) == 0;
        b.h_tab[i] = d;
        b.h_tab[n + i] = kind == BATCH_FACE ? b.d_gray + (size_t)i * cols * rows : d;
    }
    // host frames always land at the same places: the table is only copied when it changes (device frames, a new shape)
    if (!std::equal(b.h_tab, b.h_tab + 2 * n, b.tab_last.begin(), b.tab_last.end())) {
        NV_CUDA(cudaMemcpyAsync(b.d_tab, b.h_tab, 2 * (size_t)n * sizeof(uint8_t *), cudaMemcpyHostToDevice, ctx->stream));
        b.tab_last.assign(b.h_tab, b.h_tab + 2 * n);
    }
    // the repeated shape replays as one CUDA graph; frame addresses reach it through the table, so they are not part of the key
    nv_ctx::BatchKey key;
    key.kind = kind; key.n = n; key.w = w; key.h = h; key.stride = stride; key.cols = cols; key.rows = rows; key.rtab = d_rtab;
    key.aligned = aligned; key.casc = casc->uid; key.sf = dp.scale_factor; key.mn = dp.min_neighbors; key.min_w = dp.min_w;
    key.min_h = dp.min_h; key.max_w = dp.max_w; key.max_h = dp.max_h; key.epoch = ctx->epoch; key.bgen = b.gen; key.slot = ctx->ps;
    key.slot_gen = ctx->ps->gen;
    const bool graphable = !ctx->debug && !ctx->no_graph;
    int nl = 0;
    ctx->batch_replayed = false;
    if (graphable && ctx->bexec && key == ctx->bkey) {
        NV_CUDA(cudaGraphLaunch(ctx->bexec, ctx->stream));
        nl = ctx->b_nl;
        ctx->batch_replayed = true;
    } else if (graphable && key == ctx->bkey_seen) {
        if (ctx->bexec) { cudaGraphExecDestroy(ctx->bexec); ctx->bexec = nullptr; }
        cudaGraph_t g = nullptr;
        NV_CUDA(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
        rc = batch_enqueue(ctx, casc, kind, n, w, h, stride, cols, rows, d_rtab, aligned, dp.min_neighbors, &nl);
        cudaError_t ce = cudaStreamEndCapture(ctx->stream, &g);
        if (rc != NV_OK || ce != cudaSuccess || !g) {
            if (g) cudaGraphDestroy(g);
            cudaGetLastError();
            ctx->no_graph = true;                      // capture is not possible here: stay on plain launches
            nl = 0;
            if ((rc = batch_enqueue(ctx, casc, kind, n, w, h, stride, cols, rows, d_rtab, aligned, dp.min_neighbors, &nl)) != NV_OK) return rc;
        } else {
            ce = cudaGraphInstantiate(&ctx->bexec, g, 0);
            cudaGraphDestroy(g);
            if (ce != cudaSuccess) { ctx->bexec = nullptr; nv_set_error("cudaGraphInstantiate: %s", cudaGetErrorString(ce)); return NV_ERR_CUDA; }
            ctx->bkey = key; ctx->b_nl = nl;
            NV_CUDA(cudaGraphLaunch(ctx->bexec, ctx->stream));
        }
    } else {
        ctx->bkey_seen = key;
        if ((rc = batch_enqueue(ctx, casc, kind, n, w, h, stride, cols, rows, d_rtab, aligned, dp.min_neighbors, &nl)) != NV_OK) return rc;
    }
    ctx->launches += nl;
    ctx->batch_launches = nl;
    for (int i = 0; i < n; i++) ctx->batch_src[i] = b.h_tab[i];   // device copies: what an overflow re-run in collect reads
    ctx->batch_on_device = true;
    ctx->batch_last = true;
    ctx->pending = true;
    return NV_OK;
}

static int batch_collect(nv_ctx *ctx, nv_rect *out, int cap, int *counts, int *total)
{
    if (!ctx || (cap > 0 && !out) || !counts) { nv_set_error("null argument"); return NV_ERR_ARG; }
    if (!ctx->pending || !ctx->batch_last) { nv_set_error("collect without a pending batch submit"); return NV_ERR_STATE; }
    NV_CUDA(cudaSetDevice(ctx->gpu));
    NV_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->pending = false;
    const int n = ctx->batch_n;
    int rc = NV_OK;
    if (ctx->batch_routed) {
        // headers and rectangles are in the mapped result blocks; an image whose grouping ran out of room runs again alone
        const long long launches0 = ctx->launches;
        ctx->batch_out.clear();
        const PlanDev &P = ctx->ps->plan;
        std::vector<nv_rect> rects;
        std::vector<int> cnt(n);
        for (int i = 0; i < n && rc == NV_OK; i++) {
            const uint8_t *blk = ctx->b.h_result + (size_t)i * BATCH_RESULT_BYTES;
            const ResultHeader *hd = reinterpret_cast<const ResultHeader *>(blk);
            if (!hd->overflow) {
                const nv_rect *r = reinterpret_cast<const nv_rect *>(blk + sizeof(ResultHeader));
                rects.insert(rects.end(), r, r + hd->n_out);
                cnt[i] = hd->n_out;
                ctx->batch_sum[0] += P.total_windows; ctx->batch_sum[1] += hd->n_alive; ctx->batch_sum[2] += hd->n_cand;
                continue;
            }
            // the re-run reads the image's device copy (or the caller's device frame); batch_single appends to batch_out
            ctx->batch_out.clear();
            if ((rc = batch_single(ctx, i, ctx->batch_src[i], true)) != NV_OK) break;
            rects.insert(rects.end(), ctx->batch_out.begin(), ctx->batch_out.end());
            cnt[i] = ctx->batch_counts[i];
        }
        ctx->batch_last = true;
        ctx->batch_launches += ctx->launches - launches0;
        if (rc != NV_OK) return rc;
        ctx->batch_out.swap(rects);
        ctx->batch_counts.swap(cnt);
    }
    const int sum = (int)ctx->batch_out.size(), m = std::min(sum, std::max(cap, 0));
    if (m > 0) memcpy(out, ctx->batch_out.data(), (size_t)m * sizeof(nv_rect));
    for (int i = 0; i < n; i++) counts[i] = ctx->batch_counts[i];
    if (total) *total = m;
    if (sum > cap) { nv_set_error("%d rectangles, caller capacity %d", sum, cap); return NV_ERR_CAPACITY; }
    return NV_OK;
}

extern "C" int nv_face_submit_batch(nv_ctx *ctx, const nv_cascade *c, const uint8_t *const *frames, int n, int width, int height,
                                    int stride_bytes, int on_device, const nv_face_params *p)
{
    int rc = batch_check(ctx, c, frames, n, width, height, stride_bytes, 3, p);
    if (rc != NV_OK) return rc;
    return batch_submit(ctx, const_cast<nv_cascade *>(c), BATCH_FACE, frames, n, width, height, stride_bytes, on_device != 0, p, nullptr);
}

extern "C" int nv_face_collect_batch(nv_ctx *ctx, nv_rect *out, int cap, int *counts, int *total)
{
    return batch_collect(ctx, out, cap, counts, total);
}

extern "C" int nv_face_detect_batch(nv_ctx *ctx, const nv_cascade *c, const uint8_t *const *frames, int n, int width, int height,
                                    int stride_bytes, int on_device, const nv_face_params *p, nv_rect *out, int cap, int *counts, int *total)
{
    if (!counts) { nv_set_error("null argument"); return NV_ERR_ARG; }
    int rc = nv_face_submit_batch(ctx, c, frames, n, width, height, stride_bytes, on_device, p);
    if (rc != NV_OK) return rc;
    return batch_collect(ctx, out, cap, counts, total);
}

extern "C" int nv_detect_multiscale_batch(nv_ctx *ctx, const nv_cascade *c, const uint8_t *const *frames, int n, int width, int height,
                                          int stride_bytes, int on_device, const nv_detect_params *p, nv_rect *out, int cap, int *counts)
{
    if (!counts) { nv_set_error("null argument"); return NV_ERR_ARG; }
    int rc = batch_check(ctx, c, frames, n, width, height, stride_bytes, 1, p);
    if (rc != NV_OK) return rc;
    if ((rc = batch_submit(ctx, const_cast<nv_cascade *>(c), BATCH_GRAY, frames, n, width, height, stride_bytes, on_device != 0, nullptr, p)) != NV_OK)
        return rc;
    return batch_collect(ctx, out, cap, counts, nullptr);
}

// ------------------------------------------------------------------------------------------------
// standalone image ops (host in, host out) for the nested elements
// ------------------------------------------------------------------------------------------------
static int upload(nv_ctx *ctx, const uint8_t *src, size_t bytes)
{
    if (bytes > ctx->frame_cap) { nv_set_error("image larger than the context"); return NV_ERR_CAPACITY; }
    NV_CUDA(cudaSetDevice(ctx->gpu));
    if (ctx->pending) { NV_CUDA(cudaStreamSynchronize(ctx->stream)); }
    return nv_h2d(ctx, src, bytes);
}

static int download(nv_ctx *ctx, const uint8_t *d_src, int row_bytes, int rows, uint8_t *dst, int dstride)
{
    NV_CUDA(cudaMemcpy2DAsync(dst, dstride, d_src, row_bytes, row_bytes, rows, cudaMemcpyDeviceToHost, ctx->stream));
    NV_CUDA(cudaStreamSynchronize(ctx->stream));
    return NV_OK;
}

extern "C" int nv_yuv2bgr(nv_ctx *ctx, const nv_yuv_frame *f, uint8_t *dst_bgr, int dst_stride)
{
    FaceSrc src;
    int rc = check_yuv(ctx, f, &src);
    if (rc != NV_OK) return rc;
    if (!dst_bgr || dst_stride < 3 * f->width) { nv_set_error("bad destination"); return NV_ERR_ARG; }
    NV_CUDA(cudaSetDevice(ctx->gpu));
    if (ctx->pending) { NV_CUDA(cudaStreamSynchronize(ctx->stream)); }
    SrcPlanes planes = {src.p[0], src.p[1], src.p[2], src.s[0], src.s[1], src.s[2]};
    if (!src.on_device && (rc = yuv_h2d(ctx, src, f->height, &planes)) != NV_OK) return rc;
    if ((rc = ensure(&ctx->d_aux, &ctx->aux_cap, (size_t)f->width * f->height * 3)) != NV_OK) return rc;
    NV_CUDA(launch_yuv2bgr(src.fmt, planes, f->width, f->height, ctx->d_aux, 3 * f->width, ctx->stream));
    ctx->launches += 1;
    return download(ctx, ctx->d_aux, 3 * f->width, f->height, dst_bgr, dst_stride);
}

extern "C" int nv_bgr2gray(nv_ctx *ctx, const uint8_t *src, int width, int height, int stride_bytes, int channels,
                           uint8_t *dst_gray, int dst_stride)
{
    if (channels != 3 && channels != 4) { nv_set_error("channels must be 3 or 4"); return NV_ERR_ARG; }
    int rc = check_frame(ctx, src, width, height, stride_bytes, channels);
    if (rc != NV_OK) return rc;
    if (!dst_gray || dst_stride < width) { nv_set_error("bad destination"); return NV_ERR_ARG; }
    if ((rc = upload(ctx, src, (size_t)stride_bytes * height)) != NV_OK) return rc;
    NV_CUDA(launch_bgr2gray(ctx->d_frame, width, height, stride_bytes, channels, ctx->d_gray, width, ctx->stream));
    ctx->launches++;
    return download(ctx, ctx->d_gray, width, height, dst_gray, dst_stride);
}

extern "C" int nv_equalize_hist(nv_ctx *ctx, const uint8_t *src, int width, int height, int stride_bytes, uint8_t *dst,
                                int dst_stride)
{
    int rc = check_frame(ctx, src, width, height, stride_bytes, 1);
    if (rc != NV_OK) return rc;
    if (!dst || dst_stride < width) { nv_set_error("bad destination"); return NV_ERR_ARG; }
    if ((rc = upload(ctx, src, (size_t)stride_bytes * height)) != NV_OK) return rc;
    NV_CUDA(launch_hist(ctx->d_frame, width, height, stride_bytes, ctx->d_hist, ctx->stream, ctx->d_lut));
    NV_CUDA(launch_apply_lut(ctx->d_frame, width, height, stride_bytes, ctx->d_lut, ctx->d_gray, width, ctx->stream));
    ctx->launches += 2;
    return download(ctx, ctx->d_gray, width, height, dst, dst_stride);
}

extern "C" int nv_resize_linear(nv_ctx *ctx, const uint8_t *src, int width, int height, int stride_bytes, int channels,
                                uint8_t *dst, int dst_width, int dst_height, int dst_stride)
{
    if (channels < 1 || channels > 4) { nv_set_error("channels must be 1..4"); return NV_ERR_ARG; }
    int rc = check_frame(ctx, src, width, height, stride_bytes, channels);
    if (rc != NV_OK) return rc;
    if (!dst || dst_width <= 0 || dst_height <= 0 || dst_stride < dst_width * channels) { nv_set_error("bad destination"); return NV_ERR_ARG; }
    if ((rc = upload(ctx, src, (size_t)stride_bytes * height)) != NV_OK) return rc;
    const int *d_rtab;
    if ((rc = nv_get_rtab(ctx, width, height, dst_width, dst_height, &d_rtab)) != NV_OK) return rc;
    if ((rc = ensure(&ctx->d_aux, &ctx->aux_cap, (size_t)dst_width * dst_height * channels)) != NV_OK) return rc;
    NV_CUDA(launch_resize_linear(ctx->d_frame, width, height, stride_bytes, channels, ctx->d_aux, dst_width, dst_height,
                                 dst_width * channels, d_rtab, ctx->stream));
    ctx->launches++;
    return download(ctx, ctx->d_aux, dst_width * channels, dst_height, dst, dst_stride);
}

extern "C" int nv_flip_horizontal(nv_ctx *ctx, const uint8_t *src, int width, int height, int stride_bytes, uint8_t *dst,
                                  int dst_stride)
{
    int rc = check_frame(ctx, src, width, height, stride_bytes, 1);
    if (rc != NV_OK) return rc;
    if (!dst || dst_stride < width) { nv_set_error("bad destination"); return NV_ERR_ARG; }
    if ((rc = upload(ctx, src, (size_t)stride_bytes * height)) != NV_OK) return rc;
    NV_CUDA(launch_flip(ctx->d_frame, width, height, stride_bytes, ctx->d_gray, width, ctx->stream));
    ctx->launches++;
    return download(ctx, ctx->d_gray, width, height, dst, dst_stride);
}

// ------------------------------------------------------------------------------------------------
// tracker
// ------------------------------------------------------------------------------------------------
#define TRK_MAX_COMPONENTS 16384

// gstnubotracker.cpp:119-200 — host-side, a handful of rectangles
static float trk_calc_dist(const nv_rect &a, const nv_rect &b)
{
    int c1x = a.x + a.width / 2, c1y = a.y + a.height / 2, c2x = b.x + b.width / 2, c2y = b.y + b.height / 2;
    return (float)sqrt((double)((c1x - c2x) * (c1x - c2x) + (c1y - c2y) * (c1y - c2y)));
}
static bool trk_inside(int px, int py, const nv_rect &r)
{
    return r.x <= px && px < r.x + r.width && r.y <= py && py < r.y + r.height;
}
static nv_rect trk_merge(const nv_rect &r1, const nv_rect &r2)
{
    int b1x = r1.x + r1.width, b1y = r1.y + r1.height, b2x = r2.x + r2.width, b2y = r2.y + r2.height;
    if (trk_inside(r2.x, r2.y, r1) && trk_inside(b2x, b2y, r1)) return r1;
    if (trk_inside(r1.x, r1.y, r2) && trk_inside(b1x, b1y, r2)) return r2;
    nv_rect o;
    o.x = std::min(r1.x, r2.x); o.y = std::min(r1.y, r2.y);
    o.width = std::max(b1x, b2x) - o.x; o.height = std::max(b1y, b2y) - o.y;
    return o;
}
static void trk_join_objects(std::vector<nv_rect> &v, int min_area, long max_area, int distance)
{
    auto area_ok = [&](const nv_rect &r) { long a = (long)r.width * r.height; return a > min_area && a < max_area; };
    for (int a = (int)v.size() - 1; a >= 0; a--) {
        if (area_ok(v[a])) {
            for (int b = a - 1; b >= 0; b--)
                if (area_ok(v[b]) && (float)distance > trk_calc_dist(v[a], v[b])) {
                    v[b] = trk_merge(v[a], v[b]);
                    v.erase(v.begin() + a);
                    break;
                }
        } else
            v.erase(v.begin() + a);
    }
}

// host-logic tap: __join_objects (TRK:171-200) on an explicit list, in place
extern "C" int nv_debug_join_objects(nv_rect *rects, int n_in, int min_area, long max_area, int distance, int *n)
{
    if (n_in < 0 || (n_in > 0 && !rects) || !n) { nv_set_error("bad argument"); return NV_ERR_ARG; }
    std::vector<nv_rect> v(rects, rects + n_in);
    trk_join_objects(v, min_area, max_area, distance);
    for (size_t i = 0; i < v.size(); i++) rects[i] = v[i];
    *n = (int)v.size();
    return NV_OK;
}

// device time of the LAST nv_tracker_process kernel on this ctx (profiling on), CUDA events on the ctx's stream
extern "C" int nv_ctx_get_tracker_kernel_ms(nv_ctx *ctx, float *ms)
{
    if (!ctx || !ms) { nv_set_error("null argument"); return NV_ERR_ARG; }
    if (!ctx->profile || !ctx->prof_set[2] || !ctx->prof_set[3]) { nv_set_error("profiling is off or no tracker call has run"); return NV_ERR_STATE; }
    NV_CUDA(cudaSetDevice(ctx->gpu));
    NV_CUDA(cudaEventSynchronize(ctx->prof_ev[3]));
    NV_CUDA(cudaEventElapsedTime(ms, ctx->prof_ev[2], ctx->prof_ev[3]));
    return NV_OK;
}

extern "C" int nv_tracker_reset(nv_ctx *ctx)
{
    if (!ctx) { nv_set_error("null ctx"); return NV_ERR_ARG; }
    ctx->trk_frames = 0;
    memset(ctx->trk_val, 0, sizeof ctx->trk_val);
    if (ctx->d_trk_hist) {
        NV_CUDA(cudaSetDevice(ctx->gpu));
        NV_CUDA(cudaMemsetAsync(ctx->d_trk_hist, 0, (size_t)ctx->trk_w * ctx->trk_h, ctx->stream));
    }
    return NV_OK;
}

// src.fmt == NV_FMT_BGR: interleaved BGRA in p[0] / s[0]; else the planes of a 4:2:0 frame (checked by the callers)
static int tracker_impl(nv_ctx *ctx, const FaceSrc &src, int width, int height, double timestamp_ms, const nv_tracker_params *p,
                        nv_rect *out, int cap, int *n)
{
    int rc;
    const uint8_t *bgra = src.p[0];
    const int stride_bytes = src.s[0];
    if (!p) { nv_set_error("null params"); return NV_ERR_ARG; }
    NV_CUDA(cudaSetDevice(ctx->gpu));
    if (ctx->pending) NV_CUDA(cudaStreamSynchronize(ctx->stream));
    size_t np = (size_t)width * height;
    if (ctx->trk_w != width || ctx->trk_h != height) {        // (re)configure: gstnubotracker.cpp:202-237
        NV_CUDA(cudaStreamSynchronize(ctx->stream));
        cudaFree(ctx->d_trk_prev); cudaFree(ctx->d_trk_hist); cudaFree(ctx->d_trk_scratch); cudaFreeHost(ctx->h_trk);
        ctx->d_trk_prev = nullptr; ctx->d_trk_hist = nullptr; ctx->d_trk_scratch = nullptr; ctx->h_trk = nullptr;
        ctx->trk_w = ctx->trk_h = 0;
        const size_t sb = tracker_scratch_bytes(width, height, &ctx->trk_lo);
        NV_CUDA(cudaMalloc(&ctx->d_trk_prev, np + 16));
        NV_CUDA(cudaMalloc(&ctx->d_trk_hist, np + 16));
        NV_CUDA(cudaMemset(ctx->d_trk_hist, 0, np + 16));
        NV_CUDA(cudaMalloc(&ctx->d_trk_scratch, sb));
        NV_CUDA(cudaMemset(ctx->d_trk_scratch + ctx->trk_lo.zero_begin, 0, ctx->trk_lo.zero_end - ctx->trk_lo.zero_begin));
        NV_CUDA(cudaMallocHost(&ctx->h_trk, (TRK_MAX_COMPONENTS + 1) * sizeof(int4)));
        memset(ctx->trk_val, 0, sizeof ctx->trk_val);
        ctx->trk_w = width; ctx->trk_h = height; ctx->trk_frames = 0;
    }
    SrcPlanes planes = {src.p[0], src.p[1], src.p[2], src.s[0], src.s[1], src.s[2]};
    if (!src.on_device) {
        if (src.fmt != NV_FMT_BGR) { if ((rc = yuv_h2d(ctx, src, height, &planes)) != NV_OK) return rc; }
        else {
            if ((rc = nv_h2d(ctx, bgra, (size_t)stride_bytes * height)) != NV_OK) return rc;
            planes.p0 = ctx->d_frame;
        }
    }
    int first = ctx->trk_frames == 0, nl = 0;
    // The motion history is stored as an index into the table of live timestamps (kernels_tracker.cu).  updateMotionHistory:
    // a silhouette pixel takes ts, any other pixel whose value is below ts - MHI_DURATION (0.2, :28) drops to 0 — so an
    // entry whose value is below `del` dies in this frame; equal float values share an entry.
    const float ts = (float)timestamp_ms, del = (float)(timestamp_ms - 0.2);
    float val[256];
    val[0] = 0.f;
    for (int k = 1; k < 256; k++) val[k] = (ctx->trk_val[k] != 0.f && !(ctx->trk_val[k] < del)) ? ctx->trk_val[k] : 0.f;
    int cur = 0;
    if (!first && ts != 0.f) {                                     // ts == 0: silhouette pixels read as "no history", like every 0
        for (int k = 1; k < 256 && !cur; k++) if (val[k] == ts) cur = k;
        for (int k = 1; k < 256 && !cur; k++) if (ctx->trk_val[k] == 0.f) cur = k;       // free BEFORE this frame: no pixel holds it
        if (!cur) { nv_set_error("more than 255 distinct timestamps inside the motion-history window"); return NV_ERR_CAPACITY; }
        val[cur] = ts;
    }
    if (ctx->profile) prof_mark(ctx, 2);                           // with profiling on: events around the tracker kernel
    NV_CUDA(launch_tracker(ctx, src.fmt, planes, width, height, first, p->threshold, cur, val, &nl));
    if (ctx->profile) prof_mark(ctx, 3);
    memcpy(ctx->trk_val, val, sizeof val);
    ctx->launches += nl;
    ctx->trk_frames++;
    int total = 0;
    std::vector<nv_rect> v;
    if (!first) {
        const int4 *d_out = reinterpret_cast<const int4 *>(ctx->d_trk_scratch + ctx->trk_lo.out);
        // count and the first 1024 rectangles: written into h_trk by the kernel's last block (mapped memory)
        NV_CUDA(cudaStreamSynchronize(ctx->stream));
        const int4 *h = reinterpret_cast<const int4 *>(ctx->h_trk);
        total = h[0].x;
        int m = std::min(total, TRK_MAX_COMPONENTS);
        if (m > 1024)
            NV_CUDA(cudaMemcpy(ctx->h_trk + (1 + 1024) * sizeof(int4), d_out + 1 + 1024, (size_t)(m - 1024) * sizeof(int4),
                               cudaMemcpyDeviceToHost));
        v.resize(m);
        for (int i = 0; i < m; i++) { v[i].x = h[1 + i].x; v[i].y = h[1 + i].y; v[i].width = h[1 + i].z; v[i].height = h[1 + i].w; }
        trk_join_objects(v, p->min_area, p->max_area, p->distance);
    } else
        NV_CUDA(cudaStreamSynchronize(ctx->stream));
    int m = std::min((int)v.size(), cap);
    if (out && m > 0) memcpy(out, v.data(), (size_t)m * sizeof(nv_rect));
    if (n) *n = m;
    if (total > TRK_MAX_COMPONENTS) { nv_set_error("more than %d motion components", TRK_MAX_COMPONENTS); return NV_ERR_CAPACITY; }
    return NV_OK;
}

extern "C" int nv_tracker_process(nv_ctx *ctx, const uint8_t *bgra, int width, int height, int stride_bytes,
                                  double timestamp_ms, const nv_tracker_params *p, nv_rect *out, int cap, int *n)
{
    int rc = check_frame(ctx, bgra, width, height, stride_bytes, 4);
    if (rc != NV_OK) return rc;
    if (stride_bytes % 4) { nv_set_error("BGRA stride must be a multiple of 4"); return NV_ERR_ARG; }
    FaceSrc src = {NV_FMT_BGR, {bgra, nullptr, nullptr}, {stride_bytes, 0, 0}, false};
    return tracker_impl(ctx, src, width, height, timestamp_ms, p, out, cap, n);
}

extern "C" int nv_tracker_process_yuv(nv_ctx *ctx, const nv_yuv_frame *f, double timestamp_ms, const nv_tracker_params *p,
                                      nv_rect *out, int cap, int *n)
{
    FaceSrc src;
    int rc = check_yuv(ctx, f, &src);
    if (rc != NV_OK) return rc;
    return tracker_impl(ctx, src, f->width, f->height, timestamp_ms, p, out, cap, n);
}

// ------------------------------------------------------------------------------------------------
// parity taps
// ------------------------------------------------------------------------------------------------
static int tap_ready(nv_ctx *ctx, int level, bool need_level)
{
    if (!ctx) { nv_set_error("null ctx"); return NV_ERR_ARG; }
    if (!ctx->ps->plan_valid) { nv_set_error("no detect call has run on this context"); return NV_ERR_STATE; }
    if (ctx->batch_last) { nv_set_error("parity taps describe single calls: the last call was a batch"); return NV_ERR_STATE; }
    if (need_level && (level < 0 || level >= ctx->ps->plan.nlevels)) { nv_set_error("level out of range"); return NV_ERR_ARG; }
    NV_CUDA(cudaSetDevice(ctx->gpu));
    NV_CUDA(cudaStreamSynchronize(ctx->stream));
    return NV_OK;
}

extern "C" int nv_debug_num_levels(nv_ctx *ctx) { return ctx && ctx->ps->plan_valid && !ctx->batch_last ? ctx->ps->plan.nlevels : 0; }

extern "C" int nv_debug_level_info(nv_ctx *ctx, int level, nv_level_info *info)
{
    if (!ctx || !info || !ctx->ps->plan_valid || level < 0 || level >= ctx->ps->plan.nlevels) { nv_set_error("bad argument"); return NV_ERR_ARG; }
    if (ctx->batch_last) { nv_set_error("parity taps describe single calls: the last call was a batch"); return NV_ERR_STATE; }
    const LevelDesc &L = ctx->ps->plan.lv[level];
    info->scale = L.scale; info->width = L.lw; info->height = L.lh; info->ystep = L.ystep; info->nx = L.nx; info->ny = L.ny;
    return NV_OK;
}

extern "C" int nv_debug_get_gray(nv_ctx *ctx, uint8_t *dst, int cap_bytes, int *width, int *height)
{
    int rc = tap_ready(ctx, 0, false);
    if (rc != NV_OK) return rc;
    int W = ctx->ps->plan.W, H = ctx->ps->plan.H;
    if (width) *width = W;
    if (height) *height = H;
    if (!dst || cap_bytes < W * H) { nv_set_error("destination too small"); return NV_ERR_ARG; }
    uint8_t lut[256];
    NV_CUDA(cudaMemcpy2D(dst, W, ctx->tap_gray, ctx->tap_stride, W, H, cudaMemcpyDeviceToHost));
    NV_CUDA(cudaMemcpy(lut, ctx->tap_lut, 256, cudaMemcpyDeviceToHost));
    for (int i = 0; i < W * H; i++) dst[i] = lut[dst[i]];
    return NV_OK;
}

extern "C" int nv_debug_get_integral(nv_ctx *ctx, int level, int32_t *sum, uint32_t *sqsum)
{
    int rc = tap_ready(ctx, level, true);
    if (rc != NV_OK) return rc;
    const LevelDesc &L = ctx->ps->plan.lv[level];
    size_t ne = (size_t)L.ipitch * (L.lh + 1);
    std::vector<uint32_t> tmp(ne);
    for (int a = 0; a < 2; a++) {
        uint32_t *dst = a == 0 ? reinterpret_cast<uint32_t *>(sum) : sqsum;
        if (!dst) continue;
        NV_CUDA(cudaMemcpy(tmp.data(), (a == 0 ? ctx->d_sum : ctx->d_sq) + L.iofs, ne * sizeof(uint32_t), cudaMemcpyDeviceToHost));
        for (int r = 0; r <= L.lh; r++)
            for (int c = 0; c <= L.lw; c++) {
                int pc = L.ystep == 2 ? (c & 1) * L.iplane + (c >> 1) : c;
                dst[(size_t)r * (L.lw + 1) + c] = tmp[(size_t)r * L.ipitch + pc];
            }
    }
    return NV_OK;
}

extern "C" int nv_debug_get_tilted(nv_ctx *ctx, int level, int32_t *tilted)
{
    int rc = tap_ready(ctx, level, true);
    if (rc != NV_OK) return rc;
    if (!ctx->cur_tilted || !ctx->d_tilt || !tilted) { nv_set_error("no tilted integral: the last cascade has no tilted features"); return NV_ERR_STATE; }
    const LevelDesc &L = ctx->ps->plan.lv[level];
    NV_CUDA(cudaMemcpy2D(tilted, (size_t)(L.lw + 1) * 4, ctx->d_tilt + L.iofs, (size_t)L.ipitch * 4, (size_t)(L.lw + 1) * 4, L.lh + 1,
                         cudaMemcpyDeviceToHost));
    return NV_OK;
}

extern "C" int nv_debug_get_depth_map(nv_ctx *ctx, int level, int16_t *depth)
{
    int rc = tap_ready(ctx, level, true);
    if (rc != NV_OK) return rc;
    if (!ctx->debug || !ctx->d_depth || !depth) { nv_set_error("depth maps need nv_ctx_set_debug(ctx, 1) before the detect call"); return NV_ERR_STATE; }
    const LevelDesc &L = ctx->ps->plan.lv[level];
    NV_CUDA(cudaMemcpy(depth, ctx->d_depth + L.wofs, (size_t)L.nx * L.ny * sizeof(int16_t), cudaMemcpyDeviceToHost));
    return NV_OK;
}

extern "C" int nv_debug_get_candidates(nv_ctx *ctx, nv_rect *out, int cap, int *n)
{
    int rc = tap_ready(ctx, 0, false);
    if (rc != NV_OK) return rc;
    const ResultHeader *h = reinterpret_cast<const ResultHeader *>(ctx->h_result);
    int m = std::min(std::min(h->n_cand, ctx->cand_cap), cap);
    if (out && m > 0) NV_CUDA(cudaMemcpy(out, ctx->d_cand_rects, (size_t)m * sizeof(nv_rect), cudaMemcpyDeviceToHost));
    if (n) *n = m;
    return NV_OK;
}

extern "C" int nv_debug_get_counters(nv_ctx *ctx, long long *o)
{
    if (!ctx || !o) { nv_set_error("null argument"); return NV_ERR_ARG; }
    const ResultHeader *h = reinterpret_cast<const ResultHeader *>(ctx->h_result);
    memset(o, 0, 8 * sizeof(long long));
    if (ctx->batch_last) {                                   // a batch: windows, alive windows and candidates of all its images
        for (int i = 0; i < 3; i++) o[i] = ctx->batch_sum[i];
        o[3] = ctx->batch_launches;
        o[4] = ctx->batch_replayed && ctx->batch_routed;
        return NV_OK;
    }
    o[0] = ctx->ps->plan_valid ? ctx->ps->plan.total_windows : 0;
    o[1] = h ? h->n_alive : 0;
    o[2] = h ? h->n_cand : 0;
    o[3] = ctx->launches;
    return NV_OK;
}
