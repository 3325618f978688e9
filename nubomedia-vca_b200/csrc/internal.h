// internal.h — shared declarations of libnubovca (not part of the public C ABI).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "nubovca.h"

// plans with at most this many windows (a config-1 frame, a nested ROI) skip the tile kernels: a lone tile is a 45 us
// dependent chain, the warp-per-window kernel takes every window at once (profiles/r1_v5_summary.md)
#define NV_GROUP_UF_MIN 2048        // raw candidates: above this, groupRectangles builds its components by neighbour search + union-find
#define NV_SMALL_PLAN_WINDOWS 16384
#define NV_DEEPQ_CAP NV_SMALL_PLAN_WINDOWS   // a small plan has no more windows than that
#define NV_TAILTAB_MAX_SMEM (200 * 1024)      // k_cascade_tail_tab: classifier table + window patches per block
#define NV_TAIL_BLOCK_MIN_STUMPS 64            // stages at least this wide go to the block-per-window kernel
#define NV_COLBLK 128            // physical integral columns per block of the column scan
#define NV_MAX_LEVELS 64          // level index is packed in 6 bits of a window id
#define NV_MAX_STAGES 64
#define NV_RESULT_INLINE 1024     // rects copied back with the header in one D2H
#define NV_HIST_STRIDE 260        // ints per histogram: 256 bins + the prep kernels' last-block ticket
// batched route (nv_detect_multiscale_batch, nv_face_submit_batch): raw candidates and rectangles grouped on the device per
// image; an image with more is re-run through the single-image path in collect
#define NV_BATCH_GROUP_CAP NV_RESULT_INLINE

// ----------------------------------------------------------------------------------------------
// error plumbing
// ----------------------------------------------------------------------------------------------
void nv_set_error(const char *fmt, ...);
#define NV_CUDA(call)                                                                        \
    do {                                                                                     \
        cudaError_t e_ = (call);                                                             \
        if (e_ != cudaSuccess) {                                                             \
            nv_set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            return NV_ERR_CUDA;                                                              \
        }                                                                                    \
    } while (0)

// ----------------------------------------------------------------------------------------------
// cascade model
// ----------------------------------------------------------------------------------------------
struct HostCascade {
    int win_w = 0, win_h = 0;
    std::vector<int> stage_ntrees;
    std::vector<float> stage_thr;          // raw XML thresholds
    std::vector<int> stump_feat;
    std::vector<float> stump_thr, stump_left, stump_right;
    std::vector<int> feat_rect;            // nfeatures * 12 : x,y,w,h for 3 rects (w==0: unused)
    std::vector<float> feat_weight;        // nfeatures * 3
    int n3rect = 0;
    int order_free = 0;
    // general model: weak classifiers that are trees of more than one node and/or tilted features.  general == 0: the
    // stump arrays above describe the whole cascade (and the fast kernels apply).
    int general = 0, has_tilted = 0;
    std::vector<int> tree_nnodes;          // internal nodes per weak classifier
    std::vector<int> node_feat, node_left, node_right;   // child > 0: node of the same tree; <= 0: leaf -child of the tree
    std::vector<float> node_thr, leaves;   // nnodes + 1 leaves per tree
    std::vector<uint8_t> feat_tilted;
    // LBP model (always general): a feature is one cell rect (feat_rect[12 f .. 12 f + 3]) of a 3 x 3 grid; a node holds
    // the 256-bit subset of codes that go left instead of a threshold
    int lbp = 0;
    std::vector<int> node_subset;          // 8 words per node
};

int nv_parse_cascade_xml(const char *path, HostCascade *out);   // cascade_xml.cpp

// One weak classifier as the kernels read it: 48 bytes = 3 x 16-byte loads, warp-uniform.
struct __align__(16) DevStump {
    uint32_t r[3];      // x | y<<8 | w<<16 | h<<24
    float w[3];         // w[2]==0: two-rect feature
    float thr, left, right;
    uint32_t pad[3];
};

// General model on the device (trees of more than one node and/or tilted features): see kernels_cascade.cu
struct __align__(16) GenFeat {
    uint32_t r[3];      // x | y<<8 | w<<16 | h<<24
    float w[3];         // w[2]==0: two-rect feature
    int tilted;
    int pad;
};
struct GenModel {
    const int2 *tree;   // per weak classifier: first node, first leaf
    const int4 *node;   // feature, threshold (float bits), left, right (> 0: node of the tree; <= 0: leaf -idx)
    const float *leaf;
    const GenFeat *feat;
    const uint32_t *subset;   // LBP models: 8 words per node (node.y of such a node is unused); nullptr for Haar models
};

struct DevCascade {
    int win_w, win_h, nstages, nstumps;
    int stage_first[NV_MAX_STAGES + 1];   // prefix of stump counts
    float stage_thr[NV_MAX_STAGES];       // (float)xml - 1e-5f
};

// One weak classifier as k_cascade_tail_fast reads it (one lane per classifier): corner BYTE offsets into the window's
// private (win_h+1) x (win_w+1) integral patch, integer weights, 128 * (left - right).  Inside a stage the two-rect
// classifiers come first.  Only built when the cascade holds the exactness certificates (nv_cascade::tail_fast).
struct __align__(16) TailStump {
    uint16_t o[12];     // rect 0: a, b, c, d; rect 1; rect 2 (unused for two-rect features)
    float thr;
    int16_t w1, w2;     // w0 is -1
    double d128;
    uint32_t pad[2];
};
static_assert(sizeof(TailStump) == 48, "three 16-byte loads");

struct nv_cascade {
    unsigned long long uid = 0;           // never reused (a freed cascade's ADDRESS can be): what plans and graphs are keyed by
    HostCascade h;
    std::vector<DevStump> stumps;
    DevCascade meta;
    int tail_fast = 0;                    // order-free sums + exact integer features for EVERY stage (see fill_bulk_stumps)
    std::vector<TailStump> tail_stumps;
    std::vector<double> tail_base;        // per stage: sum of the right leaves
    std::mutex mu;
    std::map<int, DevStump *> d_stumps;   // per GPU ordinal
    std::map<int, DevCascade *> d_meta;
    std::map<int, TailStump *> d_tail;
    std::map<int, double *> d_tail_base;
    std::map<int, GenModel> d_gen;        // general cascades only
};

// ----------------------------------------------------------------------------------------------
// per-frame plan (host builds it once per (size, cascade window, parameters) key)
// ----------------------------------------------------------------------------------------------
struct LevelDesc {
    float scale;
    int lw, lh;            // level image size
    int ystep;             // 1 or 2; also the column de-interleave factor of the integral layout
    int nx, ny, nxw;       // window grid (after the stripe row limit), nxw = ceil(nx/32)
    int ipitch;            // integral row pitch, elements (all planes)
    int iplane;            // plane width, elements: physical col = (c % ystep) * iplane + c / ystep
    int iofs;              // element offset of this level in the sum / sqsum buffers
    int wofs;              // offset into per-window arrays (vnf, depth)
    int bofs;              // offset into per-32-window bit-word arrays
    int xtab, ytab;        // offsets into the pyramid coefficient tables
    int pofs;              // byte offset of the u8 level image (debug)
    int rowblk0;           // first row-block (8 rows) of this level in k_pyr_rowscan's grid
    int colblk0;           // first column-block (NV_COLBLK physical cols) in k_colscan's grid (per array)
    int chunk0;            // first 32-window chunk (row-major over levels)
    int row0;              // first window row in k_stage0_rows' grid
    int dblk0;             // first block (256 diagonals) of this level in the tilted-integral kernels' grid
    int ctile0, cntx;      // k_cascade_classes: first 64x32-window tile within the ystep class, tile columns = ceil(nx/64)
    int wtile0, wntx;      // k_cascade_wide: first tile of the level within its ystep class, tile columns = ceil(nx / NV_WTX)
};

struct PlanDev {
    int nlevels;
    int W, H;              // processing-size image (the pyramid base)
    int win_w, win_h;
    int total_rowblk, total_colblk, total_chunks, total_rows, total_windows;
    int nlv2;              // levels [0, nlv2) have ystep 2, [nlv2, nlevels) ystep 1 (scales ascend)
    int ctiles2, ctiles1;  // 64x32-window tile counts of the two ystep classes
    int wtiles[2];         // k_cascade_wide: tile counts of the ystep-2 [0] / ystep-1 [1] levels (the ystep-2 levels run k_cascade_classes: 0)
    int total_dblk;        // blocks of the tilted-integral kernels
    LevelDesc lv[NV_MAX_LEVELS];
};

struct PlanKey {
    int W = 0, H = 0, win_w = 0, win_h = 0, min_w = 0, min_h = 0, max_w = 0, max_h = 0;
    double sf = 0;
    unsigned long long casc = 0;           // nv_cascade::uid: the tile / stage-0 parameter banks of a plan are built for one cascade
    bool operator==(const PlanKey &o) const {
        return W == o.W && H == o.H && win_w == o.win_w && win_h == o.win_h && min_w == o.min_w &&
               min_h == o.min_h && max_w == o.max_w && max_h == o.max_h && sf == o.sf && casc == o.casc;
    }
};

// resize tables for cv::resize(INTER_LINEAR) (element-level resize, A.2)
struct ResizeKey {
    int sw = 0, sh = 0, dw = 0, dh = 0;
    bool operator==(const ResizeKey &o) const { return sw == o.sw && sh == o.sh && dw == o.dw && dh == o.dh; }
};

// ---- k_cascade_classes parameters (passed by value as a __grid_constant__: tensor maps and the bulk
// stages' weak classifiers live in the constant bank, so they cost no load/store-unit bandwidth) ----
#define NV_BULK_MAX_STUMPS 384
#define NV_BULK_MAX_STAGES 16
#define NV_CTX 64                  // k_stage0_tiles, k_cascade_classes: tile width and height in windows
#define NV_CTY 32
#define NV_WTX 128                 // k_cascade_wide (ystep-1 levels): tile width and height in windows.  The ystep-2 levels stay on
#define NV_WTY 64                  // k_cascade_classes: two column planes per tile make a 64x64 tile 89 KB of shared memory (2800
                                   // against 2880 frames/s), and at 64x32 the interleaved ranks are 1 % ahead

// One bulk-stage weak classifier, 64 bytes, warp-uniform.  Offsets are BYTE offsets of the rect corners a, b, c, d
// from the window's origin in the shared-memory tile.
struct __align__(16) BulkStump {
    uint4 o0, o1;                  // rects 0 and 1
    uint32_t w0, w1, w2, thr;      // weights (float bits, or int32 in the exact-integer variant), node threshold (float bits)
    uint32_t d_lo, d_hi;           // order-free variant: 128 * ((double)left - (double)right)
    uint32_t left, right;          // in-order variant: leaves (float bits)
};

struct TileParams {
    BulkStump s[NV_BULK_MAX_STUMPS];
    uint4 o2[NV_BULK_MAX_STUMPS];  // rect 2 (a copy of rect 0 with weight 0 for two-rect features)
    int stage_first[NV_BULK_MAX_STAGES + 1];   // stage s (FAST order): six-load two-rect classifiers [first[s], mid6[s]),
    int stage_mid6[NV_BULK_MAX_STAGES];        // eight-load two-rect [mid6[s], mid[s]), three-rect [mid[s], first[s+1])
    int stage_mid[NV_BULK_MAX_STAGES];
    float stage_thr[NV_BULK_MAX_STAGES];
    double stage_base[NV_BULK_MAX_STAGES];     // order-free variant: sum of the stage's right leaves
    int stage_begin, stage_end;    // bulk stages [begin, end)
    int final_stage;               // 1: stage_end == nstages, survivors are candidates
    int fast;                      // 1: order-free stage sums and exact integer feature arithmetic (certificates in fill_bulk_stumps)
    int level_begin, level_end;
    int cp, rt, ps;                // tile plane geometry: columns, rows, plane stride (words)
    int kskew;                     // bank class of window (lx, ly) = (lx + kskew * ly) & 31
    const CUtensorMap *maps;       // one per level, in global memory (written by the host before launch)
    const PlanDev *plan;
    const uint32_t *bits_alive;
    const float *vnf;
    int16_t *depth;
    uint2 *tail;                   // (window id, vnf) of windows that outlive the bulk stages
    uint32_t *cand;
    int *counters;
    int tail_cap, cand_cap;
};
static_assert(sizeof(TileParams) <= 32000, "kernel parameter space is 32764 bytes");

// ---- k_stage0_tiles parameters (large plans, FAST cascades): stage 0 evaluated DENSELY on the bulk kernel's 64x32-window
// tiles — same TMA staging, same bank classes, same six / eight-load integer classifiers — writing one "failed stage 0"
// and one "valid and passes the variance test" bit per window; k_stage0_chain then runs the skip rule along every row.
#define NV_S0T_MAX_STUMPS 8
struct Stage0TileParams {
    BulkStump s[NV_S0T_MAX_STUMPS];
    uint4 o2[NV_S0T_MAX_STUMPS];
    int stage_first[2], stage_mid6[1], stage_mid[1];   // the member names class_stage reads (one stage)
    float stage_thr[1];
    double stage_base[1];
    uint4 var;                     // byte offsets of the variance rect's corners from the window origin in the tile
    int win_w, win_h;
    int level_begin, level_end;
    int cp, rt, ps, kskew;
    const CUtensorMap *maps;
    const PlanDev *plan;
    const uint32_t *sq;
    float *vnf;
    uint32_t *bits_fail, *bits_okv;
};

// ---- k_stage0_rows_p parameters: per-level corner offsets of the stage-0 classifiers, so that the whole
// address arithmetic of stage 0 is warp-uniform and lives in the constant bank ----
#define NV_S0_MAX_STUMPS 8
struct Stage0Params {
    uint4 off[NV_MAX_LEVELS][NV_S0_MAX_STUMPS][3];   // word offsets of the rect corners a, b, c, d in the level's integral layout
    int4 var[NV_MAX_LEVELS];                         // corners of the variance-normalisation rect
    int4 lv_a[NV_MAX_LEVELS];                        // row0, nxw, nx, ystep * ipitch
    int4 lv_b[NV_MAX_LEVELS];                        // iofs, wofs, bofs, unused
    float2 cf[NV_S0_MAX_STUMPS][3];                  // (w0, w1), (w2, threshold), (left, right)
    int nlevels, total_rows, n0, win_w, win_h;
    float thr0;
    const uint32_t *sum, *sq;
    float *vnf;
    uint32_t *bits_alive;
    int *counters;
    int16_t *depth;
    uint2 *queue;                                    // small plans: (window id, vnf) of every alive window goes straight to the
    int queue_cap, queue_cidx;                       // warp-per-window kernel's queue (count in counters[queue_cidx]); else nullptr
    size_t integ_stride;                             // batched launch (k_stage0_rows_p<true>): per-image strides of sum / sq,
    int win_stride, bits_stride;                     // vnf and alive bits
};
static_assert(sizeof(Stage0Params) <= 32000, "kernel parameter space is 32764 bytes");

// header of the device result block; then rects[result_cap], level weights (double)[result_cap], neighbour counts
// (int)[result_cap] — the last two are written by calls with scores on only
struct ResultHeader {
    int n_out;          // rects written after grouping + clipping
    int n_cand;         // raw candidates (before the cap)
    int n_alive;        // windows alive after stage 0 + skip rule
    int overflow;       // 1 if a capacity was hit
};

// Everything that depends on one (image size, cascade window, parameters) key.  A context keeps the last
// NV_PLAN_SLOTS of them: the nested elements run a differently sized ROI through the same context several times per
// frame, and re-deriving + re-uploading a plan costs more than the detection itself on such small images.
struct DetGraphKey {
    const void *gray = nullptr; int gstride = 0; const void *lut = nullptr; unsigned long long casc = 0;     // nv_cascade::uid
    double sf = 0; int mn = 0; unsigned long long epoch = 0; int scores = 0;
    bool operator==(const DetGraphKey &o) const {
        return gray == o.gray && gstride == o.gstride && lut == o.lut && casc == o.casc && sf == o.sf && mn == o.mn && epoch == o.epoch &&
               scores == o.scores;
    }
};
struct PlanSlot {
    PlanKey pkey;  bool plan_valid = false;
    PlanDev plan;                                            // host copy
    PlanDev *d_plan = nullptr;
    int *d_ptab = nullptr;       size_t ptab_cap = 0;       // pyramid coefficient tables
    Stage0TileParams s0t[2];  bool use_s0t = false;  int bits_words = 0;   // dense stage 0 on tiles; 32-window words of this plan
    TileParams tp[2];  Stage0Params s0p;  bool use_s0p = false;  CUtensorMap *d_maps = nullptr;  bool use_tiles = false;
    int bulk_end = 0;  unsigned long long tp_casc = 0;  int max_lw = 0;       // uid of the cascade the banks were built for (0: none)
    unsigned long long last_use = 0, buf_gen = 0;            // LRU clock; generation of the shared buffers the tensor maps point into
    unsigned long long gen = 0;                              // bumped whenever the slot's plan or parameter banks are rebuilt
    // CUDA graph of detect_enqueue on a device-resident image (the nested ROI stages replay it frame after frame)
    cudaGraphExec_t dexec = nullptr;  DetGraphKey dkey, dkey_seen;  int d_nl = 0;
};
#define NV_PLAN_SLOTS 12

// byte offsets of the tracker's per-tile scratch inside nv_ctx::d_trk_scratch (kernels_tracker.cu)
struct TrkLayout { int ntx, nty; size_t bbox, rects, out, bseed, parent, slotlist, bcount, keys, bslot, counters, edge_flag, zero_begin, zero_end; };

struct nv_ctx {
    int gpu = 0;
    int max_w = 0, max_h = 0;
    int debug = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev_done = nullptr;
    // side stream of the two-class stages: the ystep-2 and the ystep-1 levels of a frame are independent launches (stage 0 on
    // tiles, bulk stages), neither fills the GPU alone; forked and joined with events, also inside a captured graph
    cudaStream_t stream2 = nullptr;
    cudaEvent_t ev_fork[2] = {}, ev_join[2] = {};

    // pinned staging + device frame
    uint8_t *h_frame = nullptr;  size_t frame_cap = 0;     // pinned
    uint8_t *d_frame = nullptr;
    // processing-size gray (before equalisation) and its histogram / LUT
    uint8_t *d_gray = nullptr;   size_t gray_cap = 0;
    int *d_hist = nullptr;       // 256
    uint8_t *d_lut = nullptr;    // 256
    uint8_t *d_aux = nullptr;    size_t aux_cap = 0;       // scratch image for standalone ops

    // resize tables (element-level resize), small cache keyed by (src, dst) size
    // row_period > 0: the resize reads only the source rows row_a + k * row_period and the one below each (an integer
    // down-scale by 3 or more: kmsfacedetect.cpp's 640 -> 160), so only those row pairs need to reach the device
    struct RtabEntry { ResizeKey k; int *d = nullptr; int row_a = 0, row_period = 0; };
    RtabEntry rtabs[16];  int rtab_next = 0;

    // plans (see PlanSlot); ps is the one in use
    PlanSlot *slots = nullptr;  PlanSlot *ps = nullptr;  unsigned long long use_clock = 0, buf_gen = 1;
    uint32_t *d_sum = nullptr, *d_sq = nullptr;  size_t integ_cap = 0;   // elements
    uint8_t *d_pyr = nullptr;    size_t pyr_cap = 0;        // debug level images
    float *d_vnf = nullptr;      size_t win_cap = 0;
    int16_t *d_depth = nullptr;  size_t depth_cap = 0;      // debug only
    uint32_t *d_bits_ok = nullptr;  size_t bits_cap = 0;         // one "alive after stage 0" bit per window
    uint2 *d_queue = nullptr;    size_t queue_cap = 0;
    int *d_counters = nullptr;                              // [0] queue count, [1] cand count, [2] overflow
    uint32_t *d_cand = nullptr;  int cand_cap = 0;          // packed window ids
    uint32_t *d_cand_sorted = nullptr;
    int4 *d_cand_rects = nullptr;
    uint32_t *d_adj = nullptr;   size_t adj_cap = 0;  int *d_grp = nullptr;   // similarity bit-matrix, group scratch
    uint8_t *d_result = nullptr; uint8_t *h_result = nullptr;   // ResultHeader + rects (+ scores)
    int result_cap = 0;                                     // rects
    // detection scores (nv_ctx_set_scores): last-stage sum per sorted candidate, per-class maximum (order-preserving uint64)
    int scores = 0;  bool last_scores = false, scores_ready = false;
    double *d_cand_w = nullptr;  unsigned long long *d_cls_wmax = nullptr;

    // CUDA graph of the steady-state face pipeline (one launch per frame once a call shape repeats)
    struct GraphKey {
        const void *src = nullptr; int w = 0, h = 0, stride = 0, cols = 0, rows = 0; const int *rtab = nullptr;
        unsigned long long casc = 0; double sf = 0; int mn = 0, min_w = 0, min_h = 0; unsigned long long epoch = 0;
        const PlanSlot *slot = nullptr; unsigned long long slot_gen = 0;
        int fmt = 0; const void *p1 = nullptr, *p2 = nullptr; int s1 = 0, s2 = 0;      // 4:2:0 input: chroma planes
        int scores = 0;
        bool operator==(const GraphKey &o) const {
            return scores == o.scores && fmt == o.fmt && p1 == o.p1 && p2 == o.p2 && s1 == o.s1 && s2 == o.s2 && src == o.src && w == o.w && h == o.h && stride == o.stride && cols == o.cols && rows == o.rows &&
                   rtab == o.rtab && casc == o.casc && sf == o.sf && mn == o.mn && min_w == o.min_w && min_h == o.min_h &&
                   epoch == o.epoch && slot == o.slot && slot_gen == o.slot_gen;
        }
    };
    const DevStump *cur_stumps = nullptr;  const DevCascade *cur_meta = nullptr;   // device copies of the cascade in use
    const TailStump *cur_tail = nullptr;  const double *cur_tail_base = nullptr;
    GenModel cur_gen = {};  bool use_gen = false;  bool cur_tilted = false;  // general cascade in use / it has tilted features
    bool need_tilt = false;                                                  // tilted-integral buffers exist (sticky)
    uint2 *d_queue2 = nullptr;  size_t queue2_cap = 0;                       // second window queue: general cascades on large plans
    uint2 *d_deepq = nullptr;                                                // NV_DEEPQ_CAP windows that reach the block-per-window stages (small plans)
    uint32_t *d_tilt = nullptr;  size_t tilt_cap = 0;
    cudaGraphExec_t gexec = nullptr;  GraphKey gkey, gkey_seen;  int g_nl = 0;  bool no_graph = false;  unsigned g_prof_mask = 0;
    unsigned long long epoch = 1;     // bumped whenever a buffer the pipeline binds is re-allocated or re-planned

    // last-call bookkeeping (kept so that collect() can re-run a call whose candidate buffers overflowed)
    nv_cascade *last_casc = nullptr;  nv_detect_params last_params = {};  int last_W = 0, last_H = 0;
    const uint8_t *tap_gray = nullptr, *tap_lut = nullptr;  int tap_stride = 0;
    bool pending = false;
    int profile = 0;  cudaEvent_t prof_ev[NV_NUM_STAGES + 1] = {};  bool prof_set[NV_NUM_STAGES + 1] = {};
    int last_min_neighbors = 0;
    long long launches = 0;

    // batched route (nv_detect_multiscale_batch / nv_face_submit_batch): per-image buffers, grow-only, sized for bcap images
    struct Batch {
        int cap = 0;                                        // images the per-image buffers below hold
        size_t frame_bytes = 0, gray_bytes = 0, integ = 0, wins = 0, bits = 0;   // per-image sizes the buffers were made for
        uint8_t *d_frame = nullptr, *h_stage = nullptr;     // uploaded frames / pinned staging of pageable ones
        uint8_t *d_gray = nullptr, *d_lut = nullptr;  int *d_hist = nullptr;
        uint32_t *d_sum = nullptr, *d_sq = nullptr, *d_bits = nullptr;  float *d_vnf = nullptr;
        uint2 *d_queue = nullptr;  uint32_t *d_cand = nullptr, *d_sorted = nullptr;  int4 *d_rects = nullptr;
        uint32_t *d_adj = nullptr;  int *d_grp = nullptr;
        int *d_counters = nullptr;                          // 16 shared + 16 per image
        uint8_t *d_result = nullptr, *h_result = nullptr;   // per image: ResultHeader + NV_BATCH_GROUP_CAP rects
        const uint8_t **d_tab = nullptr, **h_tab = nullptr; // per call: N source frames, N gray images
        std::vector<const uint8_t *> tab_last;             // what d_tab holds
        unsigned long long gen = 1;                         // bumped whenever a buffer above moves
    } b;
    struct BatchKey {
        int kind = 0, n = 0, w = 0, h = 0, stride = 0, cols = 0, rows = 0; const int *rtab = nullptr; bool aligned = false;
        unsigned long long casc = 0; double sf = 0; int mn = 0, min_w = 0, min_h = 0, max_w = 0, max_h = 0;
        unsigned long long epoch = 0, bgen = 0; const PlanSlot *slot = nullptr; unsigned long long slot_gen = 0;
        bool operator==(const BatchKey &o) const {
            return kind == o.kind && n == o.n && w == o.w && h == o.h && stride == o.stride && cols == o.cols && rows == o.rows &&
                   rtab == o.rtab && aligned == o.aligned && casc == o.casc && sf == o.sf && mn == o.mn && min_w == o.min_w &&
                   min_h == o.min_h && max_w == o.max_w && max_h == o.max_h && epoch == o.epoch && bgen == o.bgen && slot == o.slot &&
                   slot_gen == o.slot_gen;
        }
    };
    cudaGraphExec_t bexec = nullptr;  BatchKey bkey, bkey_seen;  int b_nl = 0;
    // last batch call: what collect needs (route, images, the overflow re-run's inputs), and what the counters tap reports
    bool batch_last = false, batch_routed = false, batch_replayed = false;  int batch_n = 0, batch_kind = 0;
    std::vector<const uint8_t *> batch_src;  int batch_w = 0, batch_h = 0, batch_stride = 0;  bool batch_on_device = false;
    nv_face_params batch_fp = {};  nv_detect_params batch_dp = {};  nv_cascade *batch_casc = nullptr;
    long long batch_sum[3] = {0, 0, 0}, batch_launches = 0;
    std::vector<nv_rect> batch_out;  std::vector<int> batch_counts;      // collected rectangles (image after image) and counts

    // tracker state (gstnubotracker.cpp:88-106 priv + the file-static img_prev :108, made per-ctx)
    // d_trk_hist: the motion history as one byte per pixel, an index into trk_val (the live timestamps; 0 = no history)
    uint8_t *d_trk_prev = nullptr, *d_trk_hist = nullptr, *d_trk_scratch = nullptr;
    TrkLayout trk_lo = {};
    float trk_val[256] = {};
    int trk_w = 0, trk_h = 0;  long long trk_frames = 0;
    uint8_t *h_trk = nullptr;
};

// ----------------------------------------------------------------------------------------------
// kernel launchers (each returns cudaGetLastError())
// ----------------------------------------------------------------------------------------------
// kernels_prep.cu
struct SrcPlanes { const uint8_t *p0, *p1, *p2; int s0, s1, s2; };    // planes of a 4:2:0 frame: Y, U|UV|VU, V
cudaError_t launch_face_prep_yuv(int fmt, const SrcPlanes &s, int sw, int sh, uint8_t *gray, int dw, int dh, const int *rtab,
                                 int *hist, cudaStream_t st, uint8_t *lut = nullptr);
cudaError_t launch_yuv2bgr(int fmt, const SrcPlanes &s, int w, int h, uint8_t *dst, int dstride, cudaStream_t st);
cudaError_t launch_yuv2gray(int fmt, const SrcPlanes &s, int w, int h, uint8_t *dst, int dstride, cudaStream_t st);
// context.cu: checks a 4:2:0 frame against the ctx and makes its planes device-resident (one H2D copy when they lie in one
// block of host memory); fills the device plane pointers
int nv_yuv_upload(nv_ctx *ctx, const nv_yuv_frame *f, SrcPlanes *planes);
cudaError_t launch_face_prep(const uint8_t *src, int sw, int sh, int sstride, int cn, uint8_t *gray, int dw, int dh,
                             const int *rtab, int *hist, cudaStream_t st, uint8_t *lut = nullptr);   // lut: the last block also writes the equalizeHist LUT (hist holds 257 ints)
cudaError_t launch_bgr2gray(const uint8_t *src, int w, int h, int sstride, int cn, uint8_t *dst, int dstride,
                            cudaStream_t st);
cudaError_t launch_resize_linear(const uint8_t *src, int sw, int sh, int sstride, int cn, uint8_t *dst, int dw, int dh,
                                 int dstride, const int *rtab, cudaStream_t st);
cudaError_t launch_hist(const uint8_t *src, int w, int h, int stride, int *hist, cudaStream_t st, uint8_t *lut = nullptr);   // lut: as launch_face_prep (hist holds 257 ints)
cudaError_t launch_apply_lut(const uint8_t *src, int w, int h, int sstride, const uint8_t *lut, uint8_t *dst, int dstride,
                             cudaStream_t st);
cudaError_t launch_flip(const uint8_t *src, int w, int h, int sstride, uint8_t *dst, int dstride, cudaStream_t st);
// host-side table builders (exact OpenCV coefficient arithmetic)
void build_resize_tables(int sw, int sh, int dw, int dh, std::vector<int> &tab);
// layout of rtab: [0]=mode(0 copy,1 box2,2 linear); then xofs[dw], xa[dw] (a0 | a1<<16), y0[dh], y1[dh], yb[dh]
enum { RT_COPY = 0, RT_BOX2 = 1, RT_LINEAR = 2 };

// kernels_pyramid.cu
cudaError_t launch_pyr_rowscan(const PlanDev *plan, int total_rowblk, const uint8_t *gray, int gstride, const uint8_t *lut,
                               const int *ptab, uint32_t *sum, uint32_t *sq, uint8_t *pyr_debug, cudaStream_t st);
cudaError_t launch_colscan(const PlanDev *plan, int total_colblk, uint32_t *sum, uint32_t *sq, cudaStream_t st);
cudaError_t launch_tilted(const PlanDev *plan, int total_dblk, const uint32_t *sum, uint32_t *tilt, cudaStream_t st);

// kernels_cascade.cu
cudaError_t launch_queue_stages(const PlanDev *plan, const DevCascade *meta, const DevStump *stumps, const uint32_t *sum,
                                const uint2 *queue, int *counters, uint32_t *cand, int cand_cap, int16_t *depth,
                                int nblocks, cudaStream_t st);

cudaError_t launch_stage0_rows(const PlanDev *plan, int total_rows, const DevCascade *meta, const DevStump *stumps,
                               const uint32_t *sum, const uint32_t *sq, float *vnf, uint32_t *bits_alive, int *counters,
                               int16_t *depth, cudaStream_t st);
cudaError_t launch_stage0_rows_gen(const PlanDev *plan, int total_rows, const DevCascade *meta, const GenModel &g,
                                   const uint32_t *sum, const uint32_t *sq, const uint32_t *tilt, float *vnf,
                                   uint32_t *bits_alive, int *counters, int16_t *depth, cudaStream_t st);
cudaError_t launch_queue_stages_gen(const PlanDev *plan, const DevCascade *meta, const GenModel &g, const uint32_t *sum,
                                    const uint32_t *tilt, const uint2 *queue, int *counters, uint32_t *cand, int cand_cap,
                                    int16_t *depth, int nblocks, int order_free, cudaStream_t st);
cudaError_t launch_queue_stages_gen_staged(const PlanDev *plan, const DevCascade *meta, const GenModel &g, const uint32_t *sum,
                                           const uint32_t *tilt, uint2 *queue_a, uint2 *queue_b, int qcap, int *counters,
                                           uint32_t *cand, int cand_cap, int16_t *depth, int nstages, int order_free,
                                           cudaStream_t st, int *nlaunch);
cudaError_t launch_cascade_classes(const TileParams &tp, int ntiles, cudaStream_t st);   // ystep-2 levels
cudaError_t launch_cascade_wide(const TileParams &tp, int ntiles, cudaStream_t st);      // ystep-1 levels
cudaError_t launch_stage0_rows_p(const Stage0Params &sp, cudaStream_t st);
bool fill_stage0_params(const nv_cascade *c, const PlanDev &P, Stage0Params *sp);
cudaError_t launch_cascade_tail(const PlanDev *plan, const DevCascade *meta, const DevStump *stumps, const uint32_t *sum,
                                const uint2 *tail, int *counters, uint32_t *cand, int cand_cap, int16_t *depth,
                                int stage_begin, int order_free, int nblocks, cudaStream_t st, int smem_bytes);
cudaError_t launch_alive_to_queue(const PlanDev *plan, int total_rows, const float *vnf, const uint32_t *bits_alive,
                                  uint2 *queue, int *counters, int queue_cap, cudaStream_t st, int cidx = 4);
void fill_bulk_stumps(const nv_cascade *c, int ystep, int cp, int ps, int stage_begin, int stage_end, TileParams *tp);
bool fill_stage0_tile_params(const nv_cascade *c, int ystep, int cp, int rt, int ps, int kskew, Stage0TileParams *sp);
cudaError_t launch_stage0_tiles(const Stage0TileParams &sp, int ystep, int ntiles, cudaStream_t st);
cudaError_t launch_stage0_chain(const PlanDev &plan, const uint32_t *bits_fail, const uint32_t *bits_okv,
                                uint32_t *bits_alive, int *counters, int16_t *depth, cudaStream_t st);
void build_tail_stumps(nv_cascade *c);
cudaError_t launch_cascade_tail_fast(const PlanDev *plan, const DevCascade *meta, const TailStump *tstumps, const double *tbase,
                                     const uint32_t *sum, const uint2 *tail, int *counters, uint32_t *cand, int cand_cap,
                                     int16_t *depth, int stage_begin, int stage_end, uint2 *deep, int deep_cap, cudaStream_t st,
                                     int smem_bytes);
size_t tail_tab_smem(const DevCascade &m, int stage_begin, int stage_end);
cudaError_t launch_cascade_tail_tab(const PlanDev *plan, const DevCascade *meta, const DevCascade &hmeta, const TailStump *tstumps,
                                    const double *tbase, const uint32_t *sum, const uint2 *tail, int *counters, uint32_t *cand,
                                    int cand_cap, int16_t *depth, int stage_begin, int stage_end, uint2 *deep, int deep_cap,
                                    cudaStream_t st);
cudaError_t launch_cascade_tail_block(const PlanDev *plan, const DevCascade *meta, const TailStump *tstumps, const double *tbase,
                                      const uint32_t *sum, const uint2 *queue, int *counters, int cin, uint32_t *cand, int cand_cap,
                                      int16_t *depth, int stage_begin, int skip_counter, cudaStream_t st);

// context.cu internals shared with elements.cu
int nv_detect_device(nv_ctx *ctx, nv_cascade *casc, const uint8_t *d_gray, int W, int H, int gstride, const uint8_t *d_lut,
                     const nv_detect_params *p);
int nv_collect(nv_ctx *ctx, nv_rect *out, int cap, int *n);
// kernels of the batched route (one launch each for the whole batch)
cudaError_t launch_face_prep_batch(const uint8_t *const *srcs, int n, bool aligned, int sw, int sh, int sstride, uint8_t *gray,
                                   int dw, int dh, const int *rtab, int *hist, uint8_t *lut, cudaStream_t st);
cudaError_t launch_pyramid_batch(const PlanDev *plan, int total_rowblk, int total_colblk, int n, const uint8_t *const *grays, int gstride,
                                 const uint8_t *lut, int lut_stride, const int *ptab, uint32_t *sum, uint32_t *sq, size_t integ_stride,
                                 cudaStream_t st);
cudaError_t launch_stage0_rows_p_batch(const Stage0Params &sp, int n, cudaStream_t st);
cudaError_t launch_cascade_tail_tab_batch(const PlanDev *plan, const DevCascade *meta, const DevCascade &hmeta, const TailStump *tstumps,
                                          const double *tbase, const uint32_t *sum, size_t integ_stride, const uint2 *queue, int queue_cap,
                                          int *counters, uint32_t *cand, int cand_stride, cudaStream_t st);
cudaError_t launch_group_batch(const PlanDev *plan, int n, int *counters, const uint32_t *cand, int cand_stride, int cap, uint32_t *cand_sorted,
                               int4 *cand_rects, uint32_t *adj, size_t adj_stride, int *grp, int min_neighbors, double eps, int img_w,
                               int img_h, uint8_t *result, uint8_t *host_result, size_t result_stride, cudaStream_t st);
int nv_h2d(nv_ctx *ctx, const uint8_t *src, size_t bytes);
int nv_get_rtab(nv_ctx *ctx, int sw, int sh, int dw, int dh, const int **d_tab, const nv_ctx::RtabEntry **entry = nullptr);

// kernels_group.cu
// What the candidate sort needs to evaluate each candidate's last stage (detectMultiScale3's levelWeights) and what the
// grouping needs to pass the scores on.  w == nullptr: scores off.
struct ScoreArgs {
    const DevCascade *meta;
    const DevStump *stumps;       // stump cascades (general == 0)
    GenModel g;                   // general cascades; g.subset != nullptr: LBP (no variance factor)
    int general;
    const uint32_t *sum, *sq, *tilt;
    double *w;                    // [cand_cap] weight of the candidate of rank i
    unsigned long long *cls_wmax; // [cand_cap] per class: maximum member weight, order-preserving map
};
cudaError_t launch_group(const PlanDev *plan, int *counters, const uint32_t *cand, int cand_cap, uint32_t *cand_sorted,
                         int4 *cand_rects, uint32_t *adj, int *grp, int min_neighbors, double eps, int img_w, int img_h,
                         uint8_t *result, int result_cap, int nblocks, cudaStream_t st, int *nlaunch, bool fused = false, uint8_t *host_result = nullptr,
                         const ScoreArgs *scores = nullptr);

// kernels_tracker.cu
size_t tracker_scratch_bytes(int w, int h, TrkLayout *lo);
cudaError_t launch_tracker(nv_ctx *ctx, int fmt, const SrcPlanes &src, int w, int h, int first, int thr, int cur, const float *val256,
                           int *nlaunch);

// ----------------------------------------------------------------------------------------------
// device helpers shared by the ingest kernels (kernels_prep.cu, kernels_tracker.cu): cvtColor(COLOR_YUV2BGR_*) per pixel
// ----------------------------------------------------------------------------------------------
#ifdef __CUDACC__
struct YuvTerms { int b, g, r; };                 // chroma contributions incl. the rounding half

template <int FMT>   // 1: I420 (three planes), 2: NV12 (UV interleaved), 3: NV21 (VU interleaved)
__device__ __forceinline__ YuvTerms yuv_chroma(const SrcPlanes &s, int x, int y)
{
    int u, v;
    if (FMT == 1) {
        u = s.p1[(size_t)(y >> 1) * s.s1 + (x >> 1)];
        v = s.p2[(size_t)(y >> 1) * s.s2 + (x >> 1)];
    } else {
        const uint8_t *uv = s.p1 + (size_t)(y >> 1) * s.s1 + (x & ~1);
        u = uv[FMT == 2 ? 0 : 1];
        v = uv[FMT == 2 ? 1 : 0];
    }
    u -= 128; v -= 128;
    YuvTerms t;
    t.b = (1 << 19) + 2116026 * u;
    t.g = (1 << 19) - 852492 * v - 409993 * u;
    t.r = (1 << 19) + 1673527 * v;
    return t;
}

__device__ __forceinline__ int sat_u8(int v) { return min(max(v, 0), 255); }

__device__ __forceinline__ void yuv_pixel(const SrcPlanes &s, const YuvTerms &t, int x, int y, int c3[3])
{
    int yy = max(0, (int)s.p0[(size_t)y * s.s0 + x] - 16) * 1220542;
    c3[0] = sat_u8((yy + t.b) >> 20);
    c3[1] = sat_u8((yy + t.g) >> 20);
    c3[2] = sat_u8((yy + t.r) >> 20);
}
#endif
