// elements.cu — host-side mirrors of the six reference GStreamer elements (no GStreamer needed): per-frame
// gating, ROI arithmetic, temporal smoothing and event payloads restated from the reference's
// *_process_frame / *_send_event functions, with every OpenCV call replaced by the CUDA pipeline of this
// library.  Citations: FACE = nubo_face/.../kmsfacedetect.cpp, FACES = Faces.cpp, EYE = kmseyedetect.cpp,
// MOUTH = kmsmouthdetect.cpp, NOSE = kmsnosedetect.cpp, EAR = kmseardetect.cpp, TRK = gstnubotracker.cpp.
//
// Deliberate deviations (SURVEY.md Appendix B): ROIs are clamped to the feature frame instead of letting
// cv::Mat::operator() throw (EYE:988, MOUTH:867, NOSE:869); nose does not append to /tmp/nose.log; all
// state is per element (NOSE:151-152 and TRK:108 are process-global in the reference); stdout chatter is
// dropped (FACES:63).  view-* drawing: the rectangles (face, mouth, nose, ear, tracker) are drawn into the caller's
// frame exactly as cvRectangle(.., 3, 8, 0) does; the eye element's cv::circle (EYE:1081,1095) is not drawn.
#include <math.h>
#include <stdio.h>
#include <string.h>
#include <sys/time.h>

#include <algorithm>
#include <deque>
#include <string>

#include "internal.h"

namespace {

enum Kind { K_FACE, K_EYE, K_MOUTH, K_NOSE, K_EAR, K_TRACKER };

struct Prop { const char *name; long lo, hi, def; long value; };

struct DevImg {
    uint8_t *p = nullptr;
    size_t cap = 0;
    int w = 0, h = 0;
};

inline int cv_round(double v) { return (int)lrint(v); }
inline int cv_roundf(float v) { return (int)lrintf(v); }
double g_wall_override_ms = -1;           // nv_debug_set_wall_clock_ms: tests inject the gettimeofday() of FACE:228-236,556-560
inline double wall_ms()
{
    if (g_wall_override_ms >= 0) return g_wall_override_ms;
    struct timeval t;
    gettimeofday(&t, nullptr);
    return t.tv_sec * 1000.0 + t.tv_usec / 1000.0;
}

struct TrackedFace { nv_rect r; int id; };        // BaseFace (BaseFace.cpp): rect + id, centre = x + w/2, y + h/2

}  // namespace

struct DrawSpan { int y, xa, xb; uint32_t bgr; };                  // one overlay span, xa..xb inclusive; bgr = b | g << 8 | r << 16

struct nv_element {
    Kind kind;
    std::string factory, dir;
    nv_ctx *ctx = nullptr;  int gpu = 0;
    const nv_yuv_frame *yuv = nullptr;                                  // set while a 4:2:0 buffer is being processed
    std::vector<nv_ctx *> aux;                                          // one stream each: the ROI cascades of a frame run side by side
    std::vector<Prop> props;
    nv_cascade *c_face = nullptr, *c_a = nullptr, *c_b = nullptr;     // face / (right eye, mouth, nose, "lear") / (left eye, "rear")
    // shared detector state (FACE:87-126 and the analogous priv structs)
    int num_frame = 0, num_frames_to_process = 0, num_iter = 0;
    // every custom downstream event the sink pad saw, in arrival order (the reference queues a copy of each one,
    // FACE:258-267, EYE:198-209): what __receive_event reads from a message, nothing more
    struct Field { std::string name; bool is_structure, has_type; std::string type; nv_rect rect; };
    typedef std::vector<Field> Event;
    std::deque<Event> events_queue;
    double time_events_ms = 0;
    // face
    std::vector<TrackedFace> faces_tracked;  int faces_id = 0;  int frames_with_no_detection = 0;
    // eye / mouth / nose / ear
    std::vector<nv_rect> faces, feat_a, feat_b;                        // faces; eyes_r | mouths | noses | lear ; eyes_l | rear
    int no_det_a = 0, no_det_b = 0;
    // device images
    DevImg gray, face_img, feat_img, flip_img;
    // overlays of a device-resident frame (nv_element_transform_frame_device): recorded spans, their device copy
    std::vector<DrawSpan> spans;  DrawSpan *d_spans = nullptr;  size_t d_spans_cap = 0;
    // outputs of the last frame
    std::vector<nv_meta_rect> msg;  bool pushed = false;
    std::string signal;  bool emitted = false;

    long get(const char *n) const
    {
        for (auto &p : props) if (!strcmp(p.name, n)) return p.value;
        return 0;
    }
};

namespace {

// ------------------------------------------------------------------------------------------------
// device helpers (all stream-ordered on the element's context)
// ------------------------------------------------------------------------------------------------
int img_ensure(DevImg &im, int w, int h)
{
    size_t need = (size_t)w * h;
    if (!im.p || im.cap < need) {
        if (im.p) NV_CUDA(cudaFree(im.p));
        im.p = nullptr;
        NV_CUDA(cudaMalloc(&im.p, need + 256));
        im.cap = need;
    }
    im.w = w; im.h = h;
    return NV_OK;
}

int dev_equalize(nv_ctx *ctx, DevImg &im)
{
    NV_CUDA(launch_hist(im.p, im.w, im.h, im.w, ctx->d_hist, ctx->stream, ctx->d_lut));        // histogram, and the LUT by its last block
    NV_CUDA(launch_apply_lut(im.p, im.w, im.h, im.w, ctx->d_lut, im.p, im.w, ctx->stream));   // element-wise: in place is safe
    ctx->launches += 2;
    return NV_OK;
}

int dev_resize(nv_ctx *ctx, const DevImg &src, DevImg &dst, int dw, int dh)
{
    int rc = img_ensure(dst, dw, dh);
    if (rc != NV_OK) return rc;
    const int *tab;
    if ((rc = nv_get_rtab(ctx, src.w, src.h, dw, dh, &tab)) != NV_OK) return rc;
    NV_CUDA(launch_resize_linear(src.p, src.w, src.h, src.w, 1, dst.p, dw, dh, dw, tab, ctx->stream));
    ctx->launches++;
    return NV_OK;
}

// CascadeClassifier::detectMultiScale on a (sub-)image resident on the device; blocks for the rectangles
int dev_detect(nv_ctx *ctx, nv_cascade *c, const uint8_t *d_img, int w, int h, int stride, double sf, int mn, int minw,
               int minh, std::vector<nv_rect> &out)
{
    out.clear();
    if (!c || w <= 0 || h <= 0) return NV_OK;             // empty classifier / empty ROI: no detections
    nv_detect_params p;
    p.scale_factor = sf; p.min_neighbors = mn; p.flags = 0; p.min_w = minw; p.min_h = minh; p.max_w = p.max_h = 0;
    int rc = nv_detect_device(ctx, c, d_img, w, h, stride, ctx->d_lut + 256, &p);
    if (rc != NV_OK) return rc;
    out.resize(4096);
    int n = 0;
    rc = nv_collect(ctx, out.data(), (int)out.size(), &n);
    out.resize(rc == NV_OK ? n : 0);
    return rc;
}

// The nested stage of a frame: one detectMultiScale per face ROI (two for the eye element).  Each is a chain of a
// dozen tiny dependent kernels, so they are issued on the element's auxiliary contexts (one CUDA stream each, ROI i
// always on context i % NV_ROI_STREAMS so that its cached plan and graph are found again next frame) behind an event
// on the main stream, and collected together.  The host-side merging that follows consumes them in face order.
#define NV_ROI_STREAMS 4
struct RoiJob {
    nv_cascade *c; const uint8_t *p; int w, h, stride; double sf; int mn, minw, minh;
    std::vector<nv_rect> out;
};

int run_roi_jobs(nv_element *e, std::vector<RoiJob> &jobs)
{
    if (jobs.empty()) return NV_OK;
    nv_ctx *ctx = e->ctx;
    int rc;
    while (e->aux.size() < std::min<size_t>(jobs.size(), NV_ROI_STREAMS)) {
        nv_ctx *a = nullptr;
        if ((rc = nv_ctx_create(e->gpu, 64, 64, &a)) != NV_OK) return rc;
        e->aux.push_back(a);
    }
    NV_CUDA(cudaEventRecord(ctx->ev_done, ctx->stream));              // the feature frame is complete at this point
    const size_t na = e->aux.size();
    for (size_t base = 0; base < jobs.size(); base += na) {
        size_t end = std::min(jobs.size(), base + na);
        for (size_t i = base; i < end; i++) {
            RoiJob &j = jobs[i];
            j.out.clear();
            if (!j.c || j.w <= 0 || j.h <= 0) continue;               // empty classifier / empty ROI: no detections
            nv_ctx *a = e->aux[i - base];
            NV_CUDA(cudaStreamWaitEvent(a->stream, ctx->ev_done, 0));
            nv_detect_params p;
            p.scale_factor = j.sf; p.min_neighbors = j.mn; p.flags = 0; p.min_w = j.minw; p.min_h = j.minh; p.max_w = p.max_h = 0;
            if ((rc = nv_detect_device(a, j.c, j.p, j.w, j.h, j.stride, a->d_lut + 256, &p)) != NV_OK) return rc;
        }
        for (size_t i = base; i < end; i++) {
            RoiJob &j = jobs[i];
            if (!j.c || j.w <= 0 || j.h <= 0) continue;
            j.out.resize(4096);
            int n = 0;
            rc = nv_collect(e->aux[i - base], j.out.data(), (int)j.out.size(), &n);
            j.out.resize(rc == NV_OK ? n : 0);
            if (rc != NV_OK) return rc;
        }
    }
    return NV_OK;
}

// cv::Mat::operator()(Rect) with the rectangle clamped to the image (the reference does not check)
bool clamp_roi(nv_rect &r, int W, int H)
{
    int x0 = std::max(r.x, 0), y0 = std::max(r.y, 0), x1 = std::min(r.x + r.width, W), y1 = std::min(r.y + r.height, H);
    if (x1 <= x0 || y1 <= y0) return false;
    r.x = x0; r.y = y0; r.width = x1 - x0; r.height = y1 - y0;
    return true;
}

// first step of the nested elements (EYE:949, MOUTH:836, NOSE:834, EAR:786): the full-resolution gray image, from the BGR
// frame or — for a 4:2:0 buffer — from cvtColor(COLOR_YUV2BGR_*) of its planes, per pixel
int frame_to_gray(nv_element *e, nv_ctx *ctx, const uint8_t *frame, int stride, int W, int H, uint8_t *gray)
{
    int r;
    if (e->yuv) {
        SrcPlanes pl;
        if ((r = nv_yuv_upload(ctx, e->yuv, &pl)) != NV_OK) return r;
        NV_CUDA(launch_yuv2gray(e->yuv->format, pl, W, H, gray, W, ctx->stream));
    } else {
        if ((r = nv_upload(ctx, frame, (size_t)stride * H)) != NV_OK) return r;
        NV_CUDA(launch_bgr2gray(ctx->d_frame, W, H, stride, 3, gray, W, ctx->stream));
    }
    ctx->launches++;
    return NV_OK;
}

// ------------------------------------------------------------------------------------------------
// view-* drawing, on the host: the frame is the caller's (GStreamer-mapped) memory and a handful of rectangles are
// written per frame.  cvRectangle(img, p1, p2, color, 3, 8, 0) (BASEFACE:76, MOUTH:900, NOSE:902, EAR:754, TRK:389)
// rasterises to the one-pixel outline dilated by the radius-2 diamond |dx| + |dy| <= 2 (each edge is a 3-wide band
// whose ends carry a filled radius-2 circle), clipped to the image; checked pixel by pixel against cv2.rectangle in
// tests/test_elements_cpu.py.  The colour is the cv::Scalar as the reference builds it: CV_RGB(r, g, b) = (b, g, r, 0),
// every channel of the frame is written (the tracker's BGRA alpha becomes 0, as in the reference).
// ------------------------------------------------------------------------------------------------
struct Bgr { uint8_t b, g, r; };
inline Bgr cv_rgb(int r, int g, int b) { return Bgr{(uint8_t)b, (uint8_t)g, (uint8_t)r}; }

// Frames that live in device memory: the same rasterisers run on the host, but every span they would write is recorded
// (the frame pointer is never dereferenced) and k_draw_spans writes them into the device frame afterwards.  Spans are
// made disjoint first — where two shapes overlap the later one wins, as in the sequential host drawing.
thread_local std::vector<DrawSpan> *g_span_sink = nullptr;

void fill_span(uint8_t *frame, int W, int H, int stride, int cn, int y, int xa, int xb, Bgr c)
{
    if (y < 0 || y >= H) return;
    xa = std::max(xa, 0); xb = std::min(xb, W - 1);
    if (g_span_sink) {
        if (xa <= xb) g_span_sink->push_back(DrawSpan{y, xa, xb, (uint32_t)c.b | ((uint32_t)c.g << 8) | ((uint32_t)c.r << 16)});
        return;
    }
    uint8_t *row = frame + (size_t)y * stride;
    for (int x = xa; x <= xb; x++) {
        uint8_t *px = row + (size_t)x * cn;
        px[0] = c.b; px[1] = c.g; px[2] = c.r;
        if (cn == 4) px[3] = 0;
    }
}

void draw_rectangle3(uint8_t *frame, int W, int H, int stride, int cn, int xa, int ya, int xb, int yb, Bgr c)
{
    if (!frame) return;                              // 4:2:0 buffers: the overlays are defined on BGR(A) pixels only
    const int x0 = std::min(xa, xb), x1 = std::max(xa, xb), y0 = std::min(ya, yb), y1 = std::max(ya, yb), R = 2;
    for (int y = y0 - R; y <= y1 + R; y++) {
        int dt = abs(y - y0), db = abs(y - y1);
        if (dt <= R) fill_span(frame, W, H, stride, cn, y, x0 - (R - dt), x1 + (R - dt), c);      // top edge
        if (db <= R) fill_span(frame, W, H, stride, cn, y, x0 - (R - db), x1 + (R - db), c);      // bottom edge
        if (y >= y0 && y <= y1) {                                                                  // left and right edges
            fill_span(frame, W, H, stride, cn, y, x0 - R, x0 + R, c);
            fill_span(frame, W, H, stride, cn, y, x1 - R, x1 + R, c);
        }
    }
}

// Painter's order resolved on the host: walking the recorded spans backwards, a span keeps only the parts of its row no
// later span covers.  The result is a list of disjoint spans that can be written in any order, i.e. in parallel.
void resolve_spans(const std::vector<DrawSpan> &in, std::vector<DrawSpan> &out)
{
    std::map<int, std::vector<std::pair<int, int>>> covered;      // per row: disjoint, sorted [a, b]
    out.clear();
    for (size_t k = in.size(); k-- > 0;) {
        const DrawSpan &s = in[k];
        auto &cv = covered[s.y];
        int a = s.xa;
        std::vector<std::pair<int, int>> merged;
        merged.reserve(cv.size() + 1);
        int na = s.xa, nb = s.xb;                                  // the union interval that swallows everything it touches
        for (auto &iv : cv) {
            if (iv.second < s.xa - 1 || iv.first > s.xb + 1) { merged.push_back(iv); continue; }
            if (iv.first > a) out.push_back(DrawSpan{s.y, a, std::min(iv.first - 1, s.xb), s.bgr});
            a = std::max(a, iv.second + 1);
            na = std::min(na, iv.first); nb = std::max(nb, iv.second);
        }
        if (a <= s.xb) out.push_back(DrawSpan{s.y, a, s.xb, s.bgr});
        merged.push_back({na, nb});
        std::sort(merged.begin(), merged.end());
        cv.swap(merged);
    }
}

// one warp per span; every channel of a pixel is written (BGRA: alpha becomes 0, as cvRectangle's Scalar does)
__global__ void __launch_bounds__(256) k_draw_spans(uint8_t *__restrict__ frame, int stride, int cn, const DrawSpan *__restrict__ spans, int n)
{
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= n) return;
    const DrawSpan s = spans[w];
    uint8_t *row = frame + (size_t)s.y * stride;
    for (int x = s.xa + lane; x <= s.xb; x += 32) {
        uint8_t *px = row + (size_t)x * cn;
        px[0] = (uint8_t)s.bgr; px[1] = (uint8_t)(s.bgr >> 8); px[2] = (uint8_t)(s.bgr >> 16);
        if (cn == 4) px[3] = 0;
    }
}

// writes the recorded spans into a device frame on `st` (spans travel through a small device buffer owned by the caller)
int draw_spans_device(const std::vector<DrawSpan> &raw, uint8_t *d_frame, int stride, int cn, DrawSpan **d_buf, size_t *d_cap,
                      cudaStream_t st)
{
    if (raw.empty()) return NV_OK;
    std::vector<DrawSpan> flat;
    resolve_spans(raw, flat);
    if (flat.empty()) return NV_OK;
    if (*d_cap < flat.size()) {
        if (*d_buf) NV_CUDA(cudaFree(*d_buf));
        *d_buf = nullptr; *d_cap = 0;
        const size_t cap = flat.size() * 2 + 1024;
        NV_CUDA(cudaMalloc(d_buf, cap * sizeof(DrawSpan)));
        *d_cap = cap;
    }
    // pageable source: the copy is staged by the runtime before the call returns, `flat` may die afterwards
    NV_CUDA(cudaMemcpyAsync(*d_buf, flat.data(), flat.size() * sizeof(DrawSpan), cudaMemcpyHostToDevice, st));
    const int n = (int)flat.size();
    k_draw_spans<<<(n * 32 + 255) / 256, 256, 0, st>>>(d_frame, stride, cn, *d_buf, n);
    NV_CUDA(cudaGetLastError());
    return NV_OK;
}

// cv::circle(img, c, radius, color, thickness > 1, LINE_8, 0) (EYE:1081,1095), restated from OpenCV's drawing code:
// the circle becomes a polygon (ellipse2Poly on its degree-indexed sine table, step 5 / 18 / 30 / 90 degrees by
// radius), every edge a thick line = convex quad filled by the 16.16 fixed-point scanline filler after its outline
// was traced by the fixed-point line (clipped first: the clipped end points are plotted), plus a filled circle of
// radius thickness/2 at the joints.  Checked pixel by pixel against cv2.circle in tests/test_elements_cpu.py
// (every radius 0..150, clipped by every border).
namespace cvdraw {
const int XS = 16;
const long long ONE = 1ll << XS;
struct Img { uint8_t *p; int W, H, stride, cn; Bgr c; };
struct P2 { long long x, y; };

inline void hline(const Img &im, int y, int xa, int xb) { fill_span(im.p, im.W, im.H, im.stride, im.cn, y, xa, xb, im.c); }
inline void put(const Img &im, long long x, long long y) { if (x >= 0 && x < im.W && y >= 0 && y < im.H) hline(im, (int)y, (int)x, (int)x); }

void filled_circle(const Img &im, int cx, int cy, int radius)
{
    int err = 0, dx = radius, dy = 0, plus = 1, minus = (radius << 1) - 1;
    while (dx >= dy) {
        hline(im, cy - dy, cx - dx, cx + dx); hline(im, cy + dy, cx - dx, cx + dx);
        hline(im, cy - dx, cx - dy, cx + dy); hline(im, cy + dx, cx - dy, cx + dy);
        dy++; err += plus; plus += 2;
        int mask = (err <= 0) - 1;
        err -= minus & mask; dx += mask; minus -= mask & 2;
    }
}

bool clip_line(long long Ws, long long Hs, P2 &a, P2 &b)
{
    const long long right = Ws - 1, bottom = Hs - 1;
    if (Ws <= 0 || Hs <= 0) return false;
    long long &x1 = a.x, &y1 = a.y, &x2 = b.x, &y2 = b.y;
    int c1 = (x1 < 0) + (x1 > right) * 2 + (y1 < 0) * 4 + (y1 > bottom) * 8;
    int c2 = (x2 < 0) + (x2 > right) * 2 + (y2 < 0) * 4 + (y2 > bottom) * 8;
    if ((c1 & c2) == 0 && (c1 | c2) != 0) {
        long long t;
        if (c1 & 12) { t = c1 < 8 ? 0 : bottom; x1 += (long long)((double)(t - y1) * (x2 - x1) / (y2 - y1)); y1 = t; c1 = (x1 < 0) + (x1 > right) * 2; }
        if (c2 & 12) { t = c2 < 8 ? 0 : bottom; x2 += (long long)((double)(t - y2) * (x2 - x1) / (y2 - y1)); y2 = t; c2 = (x2 < 0) + (x2 > right) * 2; }
        if ((c1 & c2) == 0 && (c1 | c2) != 0) {
            if (c1) { t = c1 == 1 ? 0 : right; y1 += (long long)((double)(t - x1) * (y2 - y1) / (x2 - x1)); x1 = t; c1 = 0; }
            if (c2) { t = c2 == 1 ? 0 : right; y2 += (long long)((double)(t - x2) * (y2 - y1) / (x2 - x1)); x2 = t; c2 = 0; }
        }
    }
    return (c1 | c2) == 0;
}

void line2(const Img &im, P2 p1, P2 p2)                           // Line2: 16.16 fixed-point end points
{
    if (!clip_line((long long)im.W << XS, (long long)im.H << XS, p1, p2)) return;
    long long dx = p2.x - p1.x, dy = p2.y - p1.y;
    long long j = dx < 0 ? -1 : 0, ax = (dx ^ j) - j, i = dy < 0 ? -1 : 0, ay = (dy ^ i) - i;
    long long x_step, y_step;
    int ecount;
    if (ax > ay) {
        dy = (dy ^ j) - j;
        if (j) { std::swap(p1, p2); }
        x_step = ONE; y_step = (dy << XS) / (ax | 1); ecount = (int)((p2.x - p1.x) >> XS);
    } else {
        dx = (dx ^ i) - i;
        if (i) { std::swap(p1, p2); }
        x_step = (dx << XS) / (ay | 1); y_step = ONE; ecount = (int)((p2.y - p1.y) >> XS);
    }
    p1.x += ONE >> 1; p1.y += ONE >> 1;
    put(im, (p2.x + (ONE >> 1)) >> XS, (p2.y + (ONE >> 1)) >> XS);
    if (ax > ay) {
        p1.x >>= XS;
        for (; ecount >= 0; ecount--) { put(im, p1.x, p1.y >> XS); p1.x++; p1.y += y_step; }
    } else {
        p1.y >>= XS;
        for (; ecount >= 0; ecount--) { put(im, p1.x >> XS, p1.y); p1.x += x_step; p1.y++; }
    }
}

void fill_convex(const Img &im, const P2 *v, int npts)              // FillConvexPoly, shift = 16, LINE_8
{
    const long long delta = ONE >> 1, delta1 = ONE >> 1, delta2 = ONE >> 1;
    struct { int idx, di; long long x, dx; int ye; } edge[2];
    int edges = npts, imin = 0;
    long long xmin = v[0].x, xmax = v[0].x, ymin = v[0].y, ymax = v[0].y;
    P2 p0 = v[npts - 1];
    for (int i = 0; i < npts; i++) {
        P2 p = v[i];
        if (p.y < ymin) { ymin = p.y; imin = i; }
        ymax = std::max(ymax, p.y); xmax = std::max(xmax, p.x); xmin = std::min(xmin, p.x);
        line2(im, p0, p);
        p0 = p;
    }
    xmin = (xmin + delta) >> XS; xmax = (xmax + delta) >> XS; ymin = (ymin + delta) >> XS; ymax = (ymax + delta) >> XS;
    if (npts < 3 || (int)xmax < 0 || (int)ymax < 0 || (int)xmin >= im.W || (int)ymin >= im.H) return;
    ymax = std::min(ymax, (long long)im.H - 1);
    edge[0].idx = edge[1].idx = imin;
    int y = (int)ymin;
    edge[0].ye = edge[1].ye = y;
    edge[0].di = 1; edge[1].di = npts - 1;
    edge[0].x = edge[1].x = -ONE;
    edge[0].dx = edge[1].dx = 0;
    do {
        for (int i = 0; i < 2; i++) {
            if (y >= edge[i].ye) {
                int idx0 = edge[i].idx, di = edge[i].di, idx = idx0 + di;
                if (idx >= npts) idx -= npts;
                for (; edges-- > 0;) {
                    int ty = (int)((v[idx].y + delta) >> XS);
                    if (ty > y) {
                        long long xs = v[idx0].x, xe = v[idx].x;
                        edge[i].ye = ty;
                        edge[i].dx = ((xe - xs) * 2 + (ty - y)) / (2 * (ty - y));
                        edge[i].x = xs;
                        edge[i].idx = idx;
                        break;
                    }
                    idx0 = idx; idx += di;
                    if (idx >= npts) idx -= npts;
                }
            }
        }
        if (edges < 0) break;
        if (y >= 0) {
            int left = 0, right = 1;
            if (edge[0].x > edge[1].x) { left = 1; right = 0; }
            int xx1 = (int)((edge[left].x + delta1) >> XS), xx2 = (int)((edge[right].x + delta2) >> XS);
            if (xx2 >= 0 && xx1 < im.W) hline(im, y, xx1, xx2);
        }
        edge[0].x += edge[0].dx; edge[1].x += edge[1].dx;
    } while (++y <= (int)ymax);
}

void thick_line(const Img &im, P2 p0, P2 p1, int thickness, int flags)
{
    const double inv = 1. / ONE;
    double dx = (p0.x - p1.x) * inv, dy = (p1.y - p0.y) * inv, r = dx * dx + dy * dy;
    const int odd = thickness & 1;
    long long th = (long long)thickness << (XS - 1);
    if (fabs(r) > 2.220446049250313e-16) {
        r = (th + odd * ONE * 0.5) / sqrt(r);
        P2 dp = {(long long)cv_round(dy * r), (long long)cv_round(dx * r)};
        P2 pt[4] = {{p0.x + dp.x, p0.y + dp.y}, {p0.x - dp.x, p0.y - dp.y}, {p1.x - dp.x, p1.y - dp.y}, {p1.x + dp.x, p1.y + dp.y}};
        fill_convex(im, pt, 4);
    }
    for (int i = 0; i < 2; i++) {
        if (flags & (i + 1))
            filled_circle(im, (int)((p0.x + (ONE >> 1)) >> XS), (int)((p0.y + (ONE >> 1)) >> XS), (int)((th + (ONE >> 1)) >> XS));
        p0 = p1;
    }
}

void circle(uint8_t *frame, int W, int H, int stride, int cn, int cx, int cy, int radius, Bgr c, int thickness)
{
    if (!frame) return;
    static const std::vector<float> sin_tab = []() {             // OpenCV's SinTable: sine of whole degrees 0..450 written with
        std::vector<float> t(451);                               // seven decimals and read back as float literals
        char buf[32];
        for (int i = 0; i <= 450; i++) {
            snprintf(buf, sizeof buf, "%.7f", sin(i * (3.141592653589793 / 180.0)));
            t[i] = (float)strtod(buf, nullptr);
        }
        return t;
    }();
    if (radius < 0) return;
    Img im = {frame, W, H, stride, cn, c};
    const P2 C = {(long long)cx * ONE, (long long)cy * ONE};
    const long long R = (long long)radius << XS;
    int d = (int)((R + (ONE >> 1)) >> XS);
    const int delta = d < 3 ? 90 : d < 10 ? 30 : d < 15 ? 18 : 5;
    std::vector<P2> v;
    P2 prev = {-1, -1};
    bool have_prev = false;
    for (int a = 0; a < 360 + delta; a += delta) {               // ellipse2Poly(center, axes, 0, 0, 360, delta)
        int ang = a > 360 ? 360 : a;
        double x = (double)R * sin_tab[450 - ang], y = (double)R * sin_tab[ang];
        double px = (double)C.x + x * (double)sin_tab[450] - y * (double)sin_tab[0];
        double py = (double)C.y + x * (double)sin_tab[0] + y * (double)sin_tab[450];
        P2 pt;
        pt.x = (long long)cv_round(px / ONE) * ONE; pt.y = (long long)cv_round(py / ONE) * ONE;
        pt.x += cv_round(px - (double)pt.x); pt.y += cv_round(py - (double)pt.y);
        if (!have_prev || pt.x != prev.x || pt.y != prev.y) { v.push_back(pt); prev = pt; have_prev = true; }
    }
    if (v.size() <= 1) v.assign(2, C);
    int flags = 3;
    P2 p0 = v[0];
    for (size_t i = 1; i < v.size(); i++) { thick_line(im, p0, v[i], thickness, flags); p0 = v[i]; flags = 2; }
}
}  // namespace cvdraw

// ------------------------------------------------------------------------------------------------
// shared logic
// ------------------------------------------------------------------------------------------------
// frame gate common to the five detectors (FACE:797-802, EYE:939-945, MOUTH:827-832, NOSE:825-830, EAR:777-782)
bool gate_runs(nv_element *e)
{
    long p = e->get("process-x-every-4-frames");
    e->num_frame++;
    return (p == 2 && e->num_frame % 2 == 1) || (p != 2 && e->num_frame <= p);
}
void gate_end(nv_element *e) { if (e->num_frame == 4) e->num_frame = 0; }       // GOP

void add_meta(nv_element *e, const char *name, const char *type, unsigned x, unsigned y, unsigned w, unsigned h)
{
    nv_meta_rect m;
    memset(&m, 0, sizeof m);
    snprintf(m.name, sizeof m.name, "%s", name);
    snprintf(m.type, sizeof m.type, "%s", type);
    m.x = x; m.y = y; m.width = w; m.height = h;
    e->msg.push_back(m);
}
void add_signal(std::string &s, unsigned x, unsigned y, unsigned w, unsigned h)
{
    char b[96];
    snprintf(b, sizeof b, "x:%u,y:%u,width:%u,height:%u;", x, y, w, h);
    s += b;
}
// g_signal_emit rate limit (FACE:228-241 and the analogous blocks)
void maybe_emit(nv_element *e, const std::string &payload, bool any, double now_ms)
{
    if (!any) return;
    double now = now_ms >= 0 ? now_ms : wall_ms();
    if (e->get("activate-events") == 1 && now - e->time_events_ms > (double)e->get("events-ms")) {
        e->time_events_ms = now;
        e->signal = payload;
        e->emitted = true;
    }
}

// __get_timestamp (FACE:658-676, EYE:662-678, ...): the message must hold a structure-typed field named "timestamp"
bool event_has_timestamp(const nv_element::Event &ev)
{
    for (auto &f : ev) if (f.name == "timestamp") return f.is_structure;
    return false;
}

// __receive_event for eye / mouth / nose (EYE:726-764, MOUTH:705-748, NOSE:702-743): pops ONE queued message whatever it
// is.  Without a timestamp it is dropped unread; otherwise __get_event_message clears the face list and walks the fields:
//   eye, nose (EYE:680-724, NOSE:648-694): every structure-typed field other than "timestamp" counts (result = true), those
//     whose "type" is "face" are kept;
//   mouth (MOUTH:655-703): only fields named "0", "1", "2", ... IN THAT ORDER are looked at (the expected number advances
//     on a name match, structure or not), so a "motion" or otherwise named field neither counts nor is read.
bool receive_faces_event(nv_element *e)
{
    if (e->get("detect-event") == 0) return true;                  // the queue is left alone (EYE:734)
    if (e->events_queue.empty()) return false;
    nv_element::Event ev = std::move(e->events_queue.front());
    e->events_queue.pop_front();
    if (!event_has_timestamp(ev)) return false;
    e->faces.clear();
    bool res = false;
    int id = 0;
    for (auto &f : ev) {
        if (f.name == "timestamp") continue;
        if (e->kind == K_MOUTH) {
            if (f.name != std::to_string(id)) continue;
            id++;
        }
        if (!f.is_structure) continue;
        if (f.has_type && f.type == "face") e->faces.push_back(f.rect);
        res = true;
    }
    if (res) e->num_frames_to_process = 10 / (5 - (int)e->get("process-x-every-4-frames"));   // NUM_FRAMES_TO_PROCESS / (5 - p)
    return res;
}
// __receive_event of the face element (FACE:711-755): pops ONE queued message; only one that carries a timestamp and a
// structure-typed "motion" field (FACE:680-709) re-arms the detector — any other message uses up this frame's pop
bool receive_motion_event(nv_element *e)
{
    if (e->get("detect-event") == 0) return true;
    if (e->events_queue.empty()) return false;
    nv_element::Event ev = std::move(e->events_queue.front());
    e->events_queue.pop_front();
    if (!event_has_timestamp(ev)) return false;
    bool motion = false;
    for (auto &f : ev) if (f.name == "motion" && f.is_structure) motion = true;
    if (motion) e->num_frames_to_process = 10;                      // NUM_FRAMES_TO_PROCESS
    return motion;
}

// ---- Faces::track_faces (FACES:78-153) ---------------------------------------------------------
int calc_distance(int x1, int y1, int x2, int y2) { return (int)sqrt(pow((double)(x2 - x1), 2) + pow((double)(y2 - y1), 2)); }
int distance_limit(int a1, int a2) { int b = std::max(a1, a2); return b > 5000 ? 8 : (b > 2500 ? 5 : 3); }     // FACES:166-181
inline int cx(const nv_rect &r) { return r.x + r.width / 2; }
inline int cy(const nv_rect &r) { return r.y + r.height / 2; }

void track_faces(std::vector<TrackedFace> &faces, int &faces_id, std::vector<TrackedFace> cf, int track_threshold,
                 int /*pos_threshold*/, int /*area_threshold*/)
{
    std::vector<TrackedFace> nv;
    for (auto &f : faces) {
        int t_distance = track_threshold, pos = -1;
        for (size_t k = 0; k < cf.size(); k++) {
            int d = calc_distance(cx(cf[k].r), cy(cf[k].r), cx(f.r), cy(f.r));
            if (t_distance > d) { pos = (int)k; t_distance = d; }
        }
        if (pos >= 0) {
            TrackedFace &c = cf[pos];
            int d = calc_distance(cx(f.r), cy(f.r), cx(c.r), cy(c.r));
            int a_old = f.r.width * f.r.height, a_new = c.r.width * c.r.height;
            if (distance_limit(a_old, a_new) < d) { c.id = f.id; nv.push_back(c); }              // moved: take the new face
            else if (15 < (abs(a_old - a_new) * 100) / a_new) {                                   // AREA_PERCENTAGE: resized
                TrackedFace t;
                t.r.x = f.r.x; t.r.y = f.r.y; t.r.width = c.r.width; t.r.height = c.r.height; t.id = f.id;
                nv.push_back(t);
            } else nv.push_back(f);                                                               // keep the old face
            cf.erase(cf.begin() + pos);
        }
    }
    for (auto &c : cf) { c.id = faces_id++; nv.push_back(c); }
    faces.swap(nv);
}

// ------------------------------------------------------------------------------------------------
// nubofacedetector (FACE:757-853 + 179-249)
// ------------------------------------------------------------------------------------------------
int face_frame(nv_element *e, uint8_t *frame, int W, int H, int stride, double now_ms, const nv_yuv_frame *yuv = nullptr)
{
    long w2p = e->get("width-to-process");
    if (w2p <= 0) { nv_set_error("width-to-process=0 divides by zero in the reference (FACE:304)"); return NV_ERR_ARG; }
    bool got = receive_motion_event(e);
    int rc = NV_OK;
    if (got || e->num_frames_to_process > 0) {
        e->num_iter++;
        if (gate_runs(e)) {
            e->num_frames_to_process--;
            nv_face_params p;
            p.width_to_process = (int)w2p;
            p.scale_factor = 1.0 + (double)e->get("multi-scale-factor") / 100.0;     // MULTI_SCALE_FACTOR, FACE:142
            p.min_neighbors = 3; p.min_w = -1; p.min_h = -1;                          // FACE:809-811
            std::vector<nv_rect> cur(4096);
            int n = 0;
            if (!e->c_face) rc = NV_OK;
            else if (yuv) rc = nv_face_detect_yuv(e->ctx, e->c_face, yuv, &p, cur.data(), (int)cur.size(), &n);
            else rc = nv_face_detect(e->ctx, e->c_face, frame, W, H, stride, &p, cur.data(), (int)cur.size(), &n);
            cur.resize(rc == NV_OK ? n : 0);
            if (!cur.empty()) {
                std::vector<TrackedFace> cf;
                int id = 0;
                for (auto &r : cur) cf.push_back({r, id++});                          // Faces(vector<Rect>&), FACES:27-39
                track_faces(e->faces_tracked, e->faces_id, cf, (int)e->get("track-threshold"),
                            (int)e->get("euclidean-distance"), (int)e->get("area-threshold"));
            } else if (e->frames_with_no_detection < 1) e->frames_with_no_detection += 1;   // MAX_NUM_FPS_WITH_NO_DETECTION
            else { e->frames_with_no_detection = 0; e->faces_tracked.clear(); }
        }
        gate_end(e);
        if (e->get("view-faces") > 0 && frame) {         // FACE:832-849 -> Faces::draw -> BASEFACE:70-82, colors[1]; BGR frames only
            // `scale` reaches Faces::draw by value AFTER process_frame replaced a useless one (frame narrower than
            // width-to-process: W / w2p == 0) by 1 (FACE:770-782); kms_face_send_event below keeps the raw quotient
            const int sc = W / (int)w2p > 0 ? W / (int)w2p : 1;
            for (auto &f : e->faces_tracked)
                draw_rectangle3(frame, W, H, stride, 3, f.r.x * sc, f.r.y * sc, (f.r.x + f.r.width - 1) * sc,
                                (f.r.y + f.r.height - 1) * sc, cv_rgb(0, 128, 255));
        }
    }
    // kms_face_send_event (FACE:179-249): runs every frame, also on skipped ones
    unsigned norm = (unsigned)(W / w2p);
    std::string s;
    for (auto &f : e->faces_tracked) {
        unsigned x = (unsigned)f.r.x * norm, y = (unsigned)f.r.y * norm, w = (unsigned)f.r.width * norm, h = (unsigned)f.r.height * norm;
        add_meta(e, "face", "face", x, y, w, h);
        add_signal(s, x, y, w, h);
    }
    e->pushed = true;
    maybe_emit(e, s, !e->faces_tracked.empty(), now_ms);
    return rc;
}

// ------------------------------------------------------------------------------------------------
// nuboeyedetector (EYE:916-1102 + 220-308)
// ------------------------------------------------------------------------------------------------
bool contain_bb(int px, int py, const nv_rect &r)       // EYE:766-776 (inclusive on both sides)
{
    return py >= r.y && py <= r.y + r.height && px >= r.x && px <= r.x + r.width;
}

// EYE:778-862, restated literally (including its index arithmetic)
void merge_eyes_current_frame(const nv_rect &face_bb, const std::vector<nv_rect> *eye_r, std::vector<nv_rect> &eyes, int scale,
                              bool eye_left)
{
    for (int i = (int)eyes.size() - 1; i > 0; i--) {
        int ecx = eyes[i].x + eyes[i].width / 2, ecy = eyes[i].y + eyes[i].height / 2;
        if (contain_bb(ecx, ecy, eyes[i - 1]) && eyes[i].width * eyes[i].height < eyes[i - 1].width * eyes[i - 1].height)
            eyes.erase(eyes.end() - i - 1);
        else {
            ecx = eyes[i - 1].x + eyes[i - 1].width / 2; ecy = eyes[i - 1].y + eyes[i - 1].height / 2;
            if (contain_bb(ecx, ecy, eyes[i]) && eyes[i - 1].width * eyes[i - 1].height < eyes[i].width * eyes[i].height)
                eyes.erase(eyes.end() - i);
        }
    }
    // eyes found at the top of the ROI are eyebrows
    for (int i = (int)eyes.size() - 1; i >= 0; i--) {
        if (i >= (int)eyes.size()) continue;
        int y_aux = face_bb.y * scale + face_bb.height * scale * 60 / 100;
        if (face_bb.y * scale + eyes[i].y < y_aux) {
            if (i == 0 && eyes.size() == 1) { if (eye_r->size() > 0 && eye_left) eyes[i].y = eye_r->at(0).y; }
            else eyes.erase(eyes.begin() + i);
        }
    }
    if (eyes.size() > 1) {
        int middle_y = face_bb.x * scale + face_bb.height * scale / 2;      // x/y swapped in the reference, kept
        int middle_x = face_bb.y * scale + face_bb.width * scale / 2;
        for (int i = (int)eyes.size() - 1; i > 0; i--) {
            int c1y = eyes[i].y + eyes[i].height / 2, c1x = eyes[i].x + eyes[i].width / 2;
            int c2y = eyes[i - 1].y + eyes[i - 1].height / 2, c2x = eyes[i - 1].x + eyes[i - 1].width / 2;
            float s1 = (float)sqrt(pow((double)(middle_x - c1x), 2) + pow((double)(middle_y - c1y), 2));
            float s2 = (float)sqrt(pow((double)(middle_x - c2x), 2) + pow((double)(middle_y - c2y), 2));
            if (s1 < s2) eyes.erase(eyes.end() - i - 1);
            else eyes.erase(eyes.end() - i);
        }
    }
    if (eye_left && eye_r->size() > 0 && eyes.size() > 0) eyes[0].y = eye_r->at(0).y;
}

// EYE:864-900 / the common shape of MOUTH:750-796 and NOSE:745-790 (those transform while merging)
// transform_2_global_coordinates (EYE:902-913)
void to_global(std::vector<nv_rect> &v, const nv_rect &fc, int scale)
{
    for (auto &q : v) { q.x = (fc.x + q.x) * scale; q.y = (fc.y + q.y) * scale; q.width = (q.width - 1) * scale; q.height = (q.height - 1) * scale; }
}

std::vector<nv_rect> merge_consecutive(std::vector<nv_rect> &cur, const std::vector<nv_rect> &prev, double limit,
                                       bool local, const nv_rect &face, int scale)
{
    std::vector<nv_rect> res;
    for (auto &o : prev) {
        int ox = o.x + o.width / 2, oy = o.y + o.height / 2;
        for (size_t j = 0; j < cur.size(); j++) {
            int nx, ny;
            if (local) {
                nx = (cur[j].x + face.x) * scale + (cur[j].width * scale) / 2;
                ny = (cur[j].y + face.y) * scale + (cur[j].height * scale) / 2;
            } else { nx = cur[j].x + cur[j].width / 2; ny = cur[j].y + cur[j].height / 2; }
            double h2 = sqrt(pow((double)(nx - ox), 2) + pow((double)(ny - oy), 2));
            if (h2 < limit) { res.push_back(o); cur.erase(cur.begin() + j); break; }       // keep the previous rect: no jitter
        }
    }
    for (auto c : cur) {
        if (local) {       // new value: move to original-image coordinates (MOUTH:782-791, NOSE:776-785)
            c.x = cv_round((double)((face.x + c.x) * scale)); c.y = cv_round((double)((face.y + c.y) * scale));
            c.width = (c.width - 1) * scale; c.height = (c.height - 1) * scale;
        }
        res.push_back(c);
    }
    return res;
}

void hold(std::vector<nv_rect> &state, int &counter, const std::vector<nv_rect> &res, int max_empty)
{
    if (res.empty()) {
        if (counter < max_empty) counter += 1;
        else { counter = 0; state.clear(); }
    } else { counter = 0; state = res; }
}

struct Scales { double o2f, o2x, f2x; };
// conf_images of eye/mouth/nose (EYE:311-341, MOUTH:285-315, NOSE:275-308): float fields read back as double
Scales detector_scales(nv_element *e, int W)
{
    float o2f = e->get("detect-event") ? (float)W / (float)W : (float)W / 160.f;       // FACE_WIDTH
    float o2x = (float)W / (float)e->get("width-to-process");
    float f2x = o2f / o2x;
    return {(double)o2f, (double)o2x, (double)f2x};
}

int eye_frame(nv_element *e, uint8_t *frame, int W, int H, int stride, double now_ms)
{
    if (e->get("width-to-process") <= 0) { nv_set_error("width-to-process must be > 0"); return NV_ERR_ARG; }
    Scales sc = detector_scales(e, W);
    nv_ctx *ctx = e->ctx;
    int rc = NV_OK;
    if (receive_faces_event(e) || e->num_frames_to_process > 0) {
        if (gate_runs(e)) {
            e->num_frames_to_process--;
            std::vector<nv_rect> res_r, res_l;
            rc = [&]() -> int {
                int r;
                if ((r = img_ensure(e->gray, W, H)) != NV_OK) return r;
                if ((r = frame_to_gray(e, ctx, frame, stride, W, H, e->gray.p)) != NV_OK) return r;     // EYE:949
                if ((r = dev_equalize(ctx, e->gray)) != NV_OK) return r;                                 // EYE:950 (full resolution)
                if (e->get("detect-event") == 0) {
                    if ((r = dev_resize(ctx, e->gray, e->face_img, cv_round(W / sc.o2f), cv_round(H / sc.o2f))) != NV_OK) return r;
                    e->faces.clear();
                    if ((r = dev_detect(ctx, e->c_face, e->face_img.p, e->face_img.w, e->face_img.h, e->face_img.w,
                                        1.0 + e->get("multi-scale-factor") / 100.0, 3, 30, 30, e->faces)) != NV_OK) return r;   // EYE:958-960
                }
                if ((r = dev_resize(ctx, e->gray, e->feat_img, cv_round(W / sc.o2x), cv_round(H / sc.o2x))) != NV_OK) return r;  // EYE:963
                if ((r = dev_equalize(ctx, e->feat_img)) != NV_OK) return r;                                                     // EYE:964
                int iscale = (int)sc.o2x;                                  // `int scale` parameters of the helpers
                std::vector<RoiJob> jobs;                                  // per face: right-eye ROI, left-eye ROI
                std::vector<nv_rect> rois;
                for (auto &f : e->faces) {
                    nv_rect ra;
                    ra.x = (int)(f.x * sc.f2x); ra.y = (int)(f.y * sc.f2x); ra.width = (int)(f.width * sc.f2x); ra.height = (int)(f.height * sc.f2x);
                    int down = cv_roundf((float)ra.height * 40 / 100), top = cv_roundf((float)ra.height * 25 / 100);   // EYE:979-980
                    nv_rect fr = {ra.x, ra.y + top, ra.width / 2, ra.height - top - down};
                    nv_rect fl = {ra.x + ra.width / 2, ra.y + top, ra.width / 2, ra.height - top - down};
                    for (int side = 0; side < 2; side++) {                  // EYE:991-993 (right), EYE:1003-1005 (left)
                        nv_rect roi = side == 0 ? fr : fl;
                        bool ok = clamp_roi(roi, e->feat_img.w, e->feat_img.h);
                        rois.push_back(roi);
                        jobs.push_back(RoiJob{ok ? (side == 0 ? e->c_a : e->c_b) : nullptr,
                                              e->feat_img.p + (ok ? (size_t)roi.y * e->feat_img.w + roi.x : 0), roi.width, roi.height,
                                              e->feat_img.w, 1.1, 2, 20, 20, {}});
                    }
                }
                if ((r = run_roi_jobs(e, jobs)) != NV_OK) return r;
                for (size_t fi = 0; fi < e->faces.size(); fi++) {
                    nv_rect fr = rois[2 * fi], fl = rois[2 * fi + 1];
                    std::vector<nv_rect> eye_r = std::move(jobs[2 * fi].out), eye_l = std::move(jobs[2 * fi + 1].out);
                    to_global(eye_r, fr, iscale);                           // EYE:1010-1011
                    to_global(eye_l, fl, iscale);
                    if (!eye_r.empty()) {
                        merge_eyes_current_frame(fr, &eye_r, eye_r, iscale, false);
                        auto m = merge_consecutive(eye_r, e->feat_a, 7, false, fr, iscale);
                        res_r.insert(res_r.end(), m.begin(), m.end());
                    }
                    if (!eye_l.empty()) {
                        merge_eyes_current_frame(fl, &res_r, eye_l, iscale, true);
                        auto m = merge_consecutive(eye_l, e->feat_b, 7, false, fl, iscale);
                        res_l.insert(res_l.end(), m.begin(), m.end());
                    }
                }
                return NV_OK;
            }();
            hold(e->feat_a, e->no_det_a, res_r, 1);                        // EYE:1034-1064
            hold(e->feat_b, e->no_det_b, res_l, 1);
        }
        gate_end(e);
        if (e->get("view-eyes") == 1) {                  // EYE:1069-1101: one circle per side, the radius of the right eye if there is one
            int radius = -1;
            if (!e->feat_a.empty()) {
                const nv_rect &q = e->feat_a[0];
                radius = cv_round((q.width + q.height) * 0.25);
                cvdraw::circle(frame, W, H, stride, 3, q.x + q.width / 2, q.y + q.height / 2, radius, Bgr{255, 0, 0}, 4);
            }
            if (!e->feat_b.empty()) {
                const nv_rect &q = e->feat_b[0];
                if (radius < 0) radius = cv_round((q.width + q.height) * 0.25);
                cvdraw::circle(frame, W, H, stride, 3, q.x + q.width / 2, q.y + q.height / 2, radius, Bgr{255, 0, 0}, 4);
            }
        }
    }
    // kms_eye_send_event (EYE:220-308): left eyes first, then right eyes
    std::string s;
    for (auto &m : e->feat_b) { add_meta(e, "eye_left", "eye", m.x, m.y, m.width, m.height); add_signal(s, m.x, m.y, m.width, m.height); }
    for (auto &m : e->feat_a) { add_meta(e, "eye_right", "eye", m.x, m.y, m.width, m.height); add_signal(s, m.x, m.y, m.width, m.height); }
    e->pushed = true;
    maybe_emit(e, s, !e->feat_a.empty() || !e->feat_b.empty(), now_ms);
    return rc;
}

// ------------------------------------------------------------------------------------------------
// nubomouthdetector (MOUTH:798-908 + 198-275) and nubonosedetector (NOSE:792-911 + 208-268)
// ------------------------------------------------------------------------------------------------
int mouth_nose_frame(nv_element *e, uint8_t *frame, int W, int H, int stride, double now_ms)
{
    if (e->get("width-to-process") <= 0) { nv_set_error("width-to-process must be > 0"); return NV_ERR_ARG; }
    const bool mouth = e->kind == K_MOUTH;
    Scales sc = detector_scales(e, W);
    nv_ctx *ctx = e->ctx;
    int rc = NV_OK;
    std::vector<nv_rect> res;
    bool processed = false;
    if (receive_faces_event(e) || e->num_frames_to_process > 0) {
        processed = true;
        if (gate_runs(e)) {
            e->num_frames_to_process--;
            rc = [&]() -> int {
                int r;
                if ((r = img_ensure(e->gray, W, H)) != NV_OK) return r;
                if ((r = frame_to_gray(e, ctx, frame, stride, W, H, e->gray.p)) != NV_OK) return r;     // MOUTH:836, NOSE:834
                if (e->get("detect-event") == 0) {
                    if ((r = dev_resize(ctx, e->gray, e->face_img, cv_round(W / sc.o2f), cv_round(H / sc.o2f))) != NV_OK) return r;
                    if ((r = dev_equalize(ctx, e->face_img)) != NV_OK) return r;
                    e->faces.clear();
                    if ((r = dev_detect(ctx, e->c_face, e->face_img.p, e->face_img.w, e->face_img.h, e->face_img.w,
                                        1.0 + e->get("multi-scale-factor") / 100.0, 2, 3, 3, e->faces)) != NV_OK) return r;   // MOUTH:845-848
                }
                if ((r = dev_resize(ctx, e->gray, e->feat_img, cv_round(W / sc.o2x), cv_round(H / sc.o2x))) != NV_OK) return r;
                if ((r = dev_equalize(ctx, e->feat_img)) != NV_OK) return r;
                int iscale = (int)sc.o2x;
                std::vector<RoiJob> jobs;
                std::vector<nv_rect> rois;
                for (auto &f : e->faces) {
                    nv_rect ra;
                    if (mouth) {                                            // MOUTH:859-867: lower part of the face
                        const int half = cv_round((double)(float)f.height / 1.8);     // (float)h / 1.8: double division
                        ra.y = (int)((f.y + half) * sc.f2x); ra.x = (int)(f.x * sc.f2x);
                        ra.height = (int)(half * sc.f2x); ra.width = (int)(f.width * sc.f2x);
                    } else {                                                // NOSE:858-869
                        const int top = cv_roundf((float)f.height * 25 / 100), down = cv_roundf((float)f.height * 10 / 100);
                        const int side = cv_roundf((float)f.width * 25 / 100);
                        ra.y = (int)((f.y + top) * sc.f2x); ra.x = (int)((f.x + side) * sc.f2x);
                        ra.height = (int)((f.height - down - top) * sc.f2x); ra.width = (int)((f.width - side) * sc.f2x);
                    }
                    if (!clamp_roi(ra, e->feat_img.w, e->feat_img.h)) continue;
                    rois.push_back(ra);
                    jobs.push_back(RoiJob{e->c_a, e->feat_img.p + (size_t)ra.y * e->feat_img.w + ra.x, ra.width, ra.height,
                                          e->feat_img.w, 1.1, 3, 1, 1, {}});            // MOUTH:870-873, NOSE:870-873
                }
                if ((r = run_roi_jobs(e, jobs)) != NV_OK) return r;
                for (size_t i = 0; i < jobs.size(); i++) {
                    std::vector<nv_rect> &found = jobs[i].out;
                    if (!found.empty()) {
                        auto m = merge_consecutive(found, e->feat_a, mouth ? 4 : 6, true, rois[i], iscale);
                        res.insert(res.end(), m.begin(), m.end());
                    }
                }
                return NV_OK;
            }();
        }
    }
    if (processed) {                     // MOUTH:883-890 / NOSE:886-893: the list is rebuilt on every non-gated-out frame
        e->feat_a = res;
        gate_end(e);
        if (e->get(mouth ? "view-mouths" : "view-noses") == 1) {        // MOUTH:895-906, NOSE:897-909: colors[j % 8]
            static const Bgr cm[8] = {cv_rgb(255, 255, 0), cv_rgb(255, 128, 0), cv_rgb(255, 0, 0), cv_rgb(255, 0, 255),
                                      cv_rgb(0, 128, 255), cv_rgb(0, 0, 255), cv_rgb(0, 255, 255), cv_rgb(0, 255, 0)};
            static const Bgr cn[8] = {cv_rgb(255, 0, 255), cv_rgb(255, 0, 0), cv_rgb(255, 255, 0), cv_rgb(255, 128, 0),
                                      cv_rgb(0, 255, 0), cv_rgb(0, 255, 255), cv_rgb(0, 128, 255), cv_rgb(0, 0, 255)};
            int j = 0;
            for (auto &m : e->feat_a) {
                // the nose element's right edge is x + width, the mouth's x + width - 1 (NOSE:903, MOUTH:901)
                draw_rectangle3(frame, W, H, stride, 3, m.x, m.y, m.x + m.width - (mouth ? 1 : 0), m.y + m.height - 1,
                                (mouth ? cm : cn)[j % 8]);
                j++;
            }
        }
    }
    std::string s;
    if (mouth) {                          // kms_mouth_send_event: faces (x int(scale_o2f)) then mouths
        unsigned norm = (unsigned)(int)sc.o2f;
        for (auto &f : e->faces) add_meta(e, "face", "face", (unsigned)f.x * norm, (unsigned)f.y * norm, (unsigned)f.width * norm, (unsigned)f.height * norm);
        for (auto &m : e->feat_a) { add_meta(e, "mouth", "mouth", m.x, m.y, m.width, m.height); add_signal(s, m.x, m.y, m.width, m.height); }
    } else
        for (auto &m : e->feat_a) { add_meta(e, "noses", "nose", m.x, m.y, m.width, m.height); add_signal(s, m.x, m.y, m.width, m.height); }
    e->pushed = true;
    maybe_emit(e, s, !e->feat_a.empty(), now_ms);
    return rc;
}

// ------------------------------------------------------------------------------------------------
// nuboeardetector (EAR:644-729, 767-822, 192-290)
// ------------------------------------------------------------------------------------------------
int ear_find(nv_element *e, const DevImg &face_img, nv_cascade *ear_cascade, double f2e, double e2o, int face_cols, int side)
{
    nv_ctx *ctx = e->ctx;
    int r;
    if ((r = dev_detect(ctx, e->c_face, face_img.p, face_img.w, face_img.h, face_img.w, 1.0 + e->get("multi-scale-factor") / 100.0,
                        2, 3, 3, e->faces)) != NV_OK) return r;                                           // EAR:656-659
    if (e->faces.empty()) return NV_OK;
    std::vector<nv_rect> &ears = side == 0 ? e->feat_a : e->feat_b;                                         // lear : rear
    if (!ears.empty()) ears.clear();
    else if (e->no_det_a < 4) e->no_det_a += 1;                                                             // MAX_NUM_FPS_WITH_NO_DETECTION
    else { e->no_det_a = 0; ears.clear(); }
    std::vector<RoiJob> jobs;
    std::vector<nv_rect> rois;
    for (auto &f : e->faces) {
        const int top = cv_roundf((float)f.height * 20 / 100), down = cv_roundf((float)f.height * 20 / 100);
        if (side == 0) {                                                                                    // LEFT_SIDE, EAR:688-697
            f.y = (int)((f.y + top) * f2e); f.x = (int)((f.x + f.width / 2) * f2e);
            f.height = (int)((f.height - down) * f2e); f.width = (int)((f.width / 2) * f2e + 50);           // EXTRA_ROI
            if (f.x + f.width > e->feat_img.w) f.width = e->feat_img.w - f.x - 1;
        } else {                                                                                            // EAR:699-707
            f.y = (int)((f.y + top) * f2e); f.x = (int)((face_cols - f.x - f.width) * f2e - 50);
            f.height = (int)((f.height - down) * f2e); f.width = (int)((f.width / 2) * f2e);
            if (f.x < 0) f.x = 0;
        }
        nv_rect roi = f;
        if (!clamp_roi(roi, e->feat_img.w, e->feat_img.h)) continue;
        rois.push_back(roi);
        jobs.push_back(RoiJob{ear_cascade, e->feat_img.p + (size_t)roi.y * e->feat_img.w + roi.x, roi.width, roi.height,
                              e->feat_img.w, 1.1, 3, 1, 1, {}});                                           // EAR:712-715
    }
    if ((r = run_roi_jobs(e, jobs)) != NV_OK) return r;
    for (size_t i = 0; i < jobs.size(); i++)
        for (auto &q : jobs[i].out) {
            const nv_rect &roi = rois[i];
            nv_rect a;
            a.x = cv_round((roi.x + q.x) * e2o); a.y = cv_round((roi.y + q.y) * e2o);
            a.width = (int)((q.width - 1) * e2o); a.height = (int)((q.height - 1) * e2o);
            ears.push_back(a);
        }
    return NV_OK;
}

int ear_frame(nv_element *e, uint8_t *frame, int W, int H, int stride, double now_ms)
{
    if (e->get("width-to-process") <= 0) { nv_set_error("width-to-process must be > 0"); return NV_ERR_ARG; }
    float f2o_f = (float)W / 160.f, e2o_f = (float)W / (float)e->get("width-to-process"), f2e_f = f2o_f / e2o_f;   // EAR:314-316
    double f2o = f2o_f, e2o = e2o_f, f2e = f2e_f;
    nv_ctx *ctx = e->ctx;
    int rc = NV_OK;
    if (gate_runs(e)) {
        e->num_frames_to_process--;
        rc = [&]() -> int {
            int r;
            if ((r = img_ensure(e->gray, W, H)) != NV_OK) return r;
            if ((r = frame_to_gray(e, ctx, frame, stride, W, H, e->gray.p)) != NV_OK) return r;             // EAR:786
            if ((r = dev_resize(ctx, e->gray, e->face_img, cv_round(W / f2o), cv_round(H / f2o))) != NV_OK) return r;
            if ((r = dev_equalize(ctx, e->face_img)) != NV_OK) return r;
            if ((r = dev_resize(ctx, e->gray, e->feat_img, cv_round(W / e2o), cv_round(H / e2o))) != NV_OK) return r;
            if ((r = dev_equalize(ctx, e->feat_img)) != NV_OK) return r;
            if ((r = ear_find(e, e->face_img, e->c_a, f2e, e2o, e->face_img.w, 0)) != NV_OK) return r;       // lecascade, LEFT_SIDE
            if ((r = img_ensure(e->flip_img, e->face_img.w, e->face_img.h)) != NV_OK) return r;
            NV_CUDA(launch_flip(e->face_img.p, e->face_img.w, e->face_img.h, e->face_img.w, e->flip_img.p, e->face_img.w, ctx->stream));   // EAR:800
            ctx->launches++;
            return ear_find(e, e->flip_img, e->c_b, f2e, e2o, e->face_img.w, 1);                             // recascade, RIGHT_SIDE
        }();
    }
    gate_end(e);
    if (e->get("view-ears") == 1) {                                     // EAR:811-817: right ears, then left ears, colors[j % 8] each
        static const Bgr ce[8] = {cv_rgb(0, 0, 255), cv_rgb(0, 128, 255), cv_rgb(0, 255, 255), cv_rgb(0, 255, 0),
                                  cv_rgb(255, 128, 0), cv_rgb(255, 255, 0), cv_rgb(255, 0, 0), cv_rgb(255, 0, 255)};
        for (auto *v : {&e->feat_b, &e->feat_a}) {
            int j = 0;
            for (auto &m : *v) { draw_rectangle3(frame, W, H, stride, 3, m.x, m.y, m.x + m.width, m.y + m.height - 1, ce[j % 8]); j++; }
        }
    }
    // kms_ear_send_event (EAR:192-290): builds the message (profile faces, right ears, left ears) but never pushes it
    std::string s;
    for (auto &f : e->faces) add_meta(e, "face_profile", "face_profile", f.x, f.y, f.width, f.height);
    for (auto &m : e->feat_b) { add_meta(e, "ear", "ear", m.x, m.y, m.width, m.height); add_signal(s, m.x, m.y, m.width, m.height); }
    for (auto &m : e->feat_a) { add_meta(e, "ear", "ear", m.x, m.y, m.width, m.height); add_signal(s, m.x, m.y, m.width, m.height); }
    e->pushed = false;
    maybe_emit(e, s, !e->feat_a.empty() || !e->feat_b.empty(), now_ms);
    e->faces.clear();                                                                                        // EAR:858
    return rc;
}

// ------------------------------------------------------------------------------------------------
// nubotracker (TRK:339-421)
// ------------------------------------------------------------------------------------------------
int tracker_frame(nv_element *e, uint8_t *frame, int W, int H, int stride, uint64_t pts_ns, double now_ms, const nv_yuv_frame *yuv = nullptr)
{
    nv_tracker_params p;
    p.threshold = (int)e->get("set_threshold"); p.min_area = (int)e->get("set_min_area");
    p.max_area = e->get("set_max_area"); p.distance = (int)e->get("set_distance");
    std::vector<nv_rect> out(16384);
    int n = 0;
    // The reference stamps the motion history with clock() in ms (TRK:349): CPU time of the PROCESS, which advances with
    // the work of every other element in it.  The buffer's presentation time is used in its place (deliberate deviation).
    double ts = (double)pts_ns / 1e6;
    int rc = yuv ? nv_tracker_process_yuv(e->ctx, yuv, ts, &p, out.data(), (int)out.size(), &n)
                 : nv_tracker_process(e->ctx, frame, W, H, stride, ts, &p, out.data(), (int)out.size(), &n);
    if (rc != NV_OK) n = 0;
    std::string s;
    bool build = e->get("set_visual_mode") > 0 || e->get("activate-events") == 1;      // TRK:383
    for (int i = 0; i < n; i++) {
        if (e->get("set_visual_mode") > 0 && frame)                    // TRK:388-389 (BGRA frames only): rec.tl() .. rec.br(), Scalar(0, 0, 255)
            draw_rectangle3(frame, W, H, stride, 4, out[i].x, out[i].y, out[i].x + out[i].width, out[i].y + out[i].height,
                            Bgr{0, 0, 255});
        add_meta(e, "object", "object", out[i].x, out[i].y, out[i].width, out[i].height);
        if (build && e->get("activate-events") == 1) add_signal(s, out[i].x, out[i].y, out[i].width, out[i].height);
    }
    e->pushed = false;                                                 // the tracker pushes no downstream event
    maybe_emit(e, s, n > 0, now_ms);
    return rc;
}

void add_props(nv_element *e, std::initializer_list<Prop> l) { for (auto &p : l) { e->props.push_back(p); e->props.back().value = p.def; } }

std::string g_missing;                    // models nv_element_create could not load (reported through nv_last_error)
nv_cascade *try_load(const std::string &dir, const char *file)
{
    nv_cascade *c = nullptr;
    std::string path = dir + "/" + file;
    if (nv_cascade_load(path.c_str(), &c) != NV_OK) {                    // the reference logs and carries on (FACE:167-171)
        g_missing += (g_missing.empty() ? "" : ", ") + path;
        return nullptr;
    }
    return c;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
extern "C" int nv_element_create(const char *factory_name, int gpu, const char *cascade_dir, nv_element **out)
{
    if (!factory_name || !out) { nv_set_error("null argument"); return NV_ERR_ARG; }
    *out = nullptr;
    static const char *names[] = {"nubofacedetector", "nuboeyedetector", "nubomouthdetector", "nubonosedetector", "nuboeardetector", "nubotracker"};
    int kind = -1;
    for (int i = 0; i < 6; i++) if (!strcmp(factory_name, names[i])) kind = i;
    if (kind < 0) { nv_set_error("unknown element factory '%s'", factory_name); return NV_ERR_ARG; }
    nv_element *e = new nv_element();
    g_missing.clear();
    e->kind = (Kind)kind; e->factory = factory_name;
    const char *env = getenv("NUBOVCA_CASCADE_DIR");
    e->dir = cascade_dir ? cascade_dir : (env ? env : "/usr/share/opencv/haarcascades");        // FACE:40
    e->gpu = gpu;                            // the CUDA context is created with the first buffer (caps are known then)
    const Prop common[] = {{"detect-event", 0, 1, 0, 0}, {"send-meta-data", 0, 1, 0, 0}, {"width-to-process", 0, 640, 320, 0},
                           {"process-x-every-4-frames", 0, 4, 4, 0}, {"multi-scale-factor", 0, 51, 25, 0},
                           {"activate-events", 0, 1, 0, 0}, {"events-ms", 0, 30000, 30001, 0}};
    auto add_common = [&](const char *view, const char *meta_name) {
        add_props(e, {{view, 0, 1, 0, 0}});
        for (auto p : common) { if (!strcmp(p.name, "send-meta-data")) p.name = meta_name; add_props(e, {p}); }
    };
    switch (e->kind) {
    case K_FACE:
        add_common("view-faces", "send-meta-data");
        for (auto &p : e->props) if (!strcmp(p.name, "width-to-process")) p.value = p.def = 160;            // FACE:26,991
        add_props(e, {{"euclidean-distance", 0, 20, 8, 0}, {"track-threshold", 0, 100, 40, 0}, {"area-threshold", 0, 1000, 500, 0}});
        e->c_face = try_load(e->dir, "haarcascade_frontalface_alt.xml");
        break;
    case K_EYE:
        add_common("view-eyes", "send-meta-data");
        e->c_face = try_load(e->dir, "haarcascade_frontalface_alt.xml");
        e->c_a = try_load(e->dir, "haarcascade_mcs_righteye.xml");                                            // eyes_rcascade, EYE:29
        e->c_b = try_load(e->dir, "haarcascade_mcs_lefteye.xml");                                             // eyes_lcascade, EYE:28
        break;
    case K_MOUTH:
        add_common("view-mouths", "send-meta-data");
        e->c_face = try_load(e->dir, "haarcascade_frontalface_alt.xml");
        e->c_a = try_load(e->dir, "haarcascade_mcs_mouth.xml");
        break;
    case K_NOSE:
        add_common("view-noses", "send-meta-data");
        e->c_face = try_load(e->dir, "haarcascade_frontalface_alt.xml");
        e->c_a = try_load(e->dir, "haarcascade_mcs_nose.xml");
        break;
    case K_EAR:
        add_common("view-ears", "meta-data");                                                                 // EAR:1006 (not send-meta-data)
        e->c_face = try_load(e->dir, "haarcascade_profileface.xml");
        e->c_a = try_load(e->dir, "haarcascade_mcs_rightear.xml");      // lecascade <- LEAR_CONF_FILE = mcs_rightear (EAR:30-31,179,186)
        e->c_b = try_load(e->dir, "haarcascade_mcs_leftear.xml");       // recascade <- REAR_CONF_FILE = mcs_leftear
        // kms_ear_detect_init (EAR:930-960) starts view_ears at -1 and never sets events_ms (zero-filled private struct)
        for (auto &p : e->props) {
            if (!strcmp(p.name, "view-ears")) p.value = p.def = -1;
            if (!strcmp(p.name, "events-ms")) p.value = p.def = 0;
        }
        break;
    case K_TRACKER:
        add_props(e, {{"set_threshold", 0, 255, 20, 0}, {"set_min_area", 0, 10000, 50, 0}, {"set_max_area", 0, 300000, 30000, 0},
                      {"set_distance", 0, 2000, 35, 0}, {"set_visual_mode", 0, 4, 0, 0}, {"activate-events", 0, 1, 0, 0},
                      {"events-ms", 0, 30000, 30001, 0}});
        break;
    }
    *out = e;
    // like the reference, a missing model is not fatal (the element then detects nothing with it) — but it is said out loud:
    // NV_OK with a non-empty nv_last_error() that names the files
    if (!g_missing.empty()) nv_set_error("warning: %s: cascade file(s) not loaded: %s", factory_name, g_missing.c_str());
    else nv_set_error("%s", "");
    return NV_OK;
}

extern "C" void nv_element_destroy(nv_element *e)
{
    if (e) for (nv_ctx *a : e->aux) nv_ctx_destroy(a);
    if (!e) return;
    if (e->ctx) { cudaSetDevice(e->ctx->gpu); cudaStreamSynchronize(e->ctx->stream); }
    for (DevImg *im : {&e->gray, &e->face_img, &e->feat_img, &e->flip_img}) cudaFree(im->p);
    cudaFree(e->d_spans);
    nv_ctx_destroy(e->ctx);
    nv_cascade_free(e->c_face); nv_cascade_free(e->c_a); nv_cascade_free(e->c_b);
    delete e;
}

extern "C" int nv_element_set_property(nv_element *e, const char *name, long value)
{
    if (!e || !name) { nv_set_error("null argument"); return NV_ERR_ARG; }
    for (auto &p : e->props)
        if (!strcmp(p.name, name)) {
            if (value < p.lo || value > p.hi) { nv_set_error("%s: %ld outside [%ld, %ld]", name, value, p.lo, p.hi); return NV_ERR_ARG; }
            if (e->kind == K_FACE && !strcmp(name, "track-threshold")) {       // reference bug kept: the setter writes
                for (auto &q : e->props) if (!strcmp(q.name, "euclidean-distance")) q.value = value;   // euclidean_threshold (FACE:548-550)
                return NV_OK;
            }
            p.value = value;
            if (!strcmp(name, "activate-events")) e->time_events_ms = wall_ms();                      // FACE:556-560
            return NV_OK;
        }
    nv_set_error("%s has no property '%s'", e->factory.c_str(), name);
    return NV_ERR_ARG;
}

extern "C" int nv_element_get_property(nv_element *e, const char *name, long *value)
{
    if (!e || !name || !value) { nv_set_error("null argument"); return NV_ERR_ARG; }
    for (auto &p : e->props) if (!strcmp(p.name, name)) { *value = p.value; return NV_OK; }
    nv_set_error("%s has no property '%s'", e->factory.c_str(), name);
    return NV_ERR_ARG;
}

extern "C" int nv_element_property_info(nv_element *e, int index, const char **name, long *minimum, long *maximum, long *default_value)
{
    if (!e || index < 0 || index >= (int)e->props.size()) { nv_set_error("no such property index"); return NV_ERR_ARG; }
    const Prop &p = e->props[index];
    if (name) *name = p.name;
    if (minimum) *minimum = p.lo;
    if (maximum) *maximum = p.hi;
    if (default_value) *default_value = p.def;
    return NV_OK;
}

extern "C" int nv_element_push_message(nv_element *e, const nv_event_field *fields, int nfields)
{
    if (!e || nfields < 0 || (nfields > 0 && !fields)) { nv_set_error("bad argument"); return NV_ERR_ARG; }
    if (e->kind == K_EAR || e->kind == K_TRACKER) return NV_OK;        // no sink_event handler of their own: events pass through
    nv_element::Event q;
    for (int i = 0; i < nfields; i++) {
        if (!fields[i].name) { nv_set_error("field without a name"); return NV_ERR_ARG; }
        q.push_back(nv_element::Field{fields[i].name, fields[i].is_structure != 0, fields[i].type != nullptr,
                                      fields[i].type ? fields[i].type : "", fields[i].rect});
    }
    e->events_queue.push_back(std::move(q));
    return NV_OK;
}

// a face message as the face element emits it (FACE:196-226): {timestamp: time{pts}, "0": face{type "face", x, y, width, height}, ...}
extern "C" int nv_element_push_faces_event(nv_element *e, const nv_rect *faces, int n)
{
    if (n < 0 || (n > 0 && !faces)) { nv_set_error("bad argument"); return NV_ERR_ARG; }
    std::vector<std::string> names(n);
    std::vector<nv_event_field> f(n + 1);
    f[0] = nv_event_field{"timestamp", 1, nullptr, {0, 0, 0, 0}};
    for (int i = 0; i < n; i++) { names[i] = std::to_string(i); f[i + 1] = nv_event_field{names[i].c_str(), 1, "face", faces[i]}; }
    return nv_element_push_message(e, f.data(), n + 1);
}

// a motion message: {timestamp: time{pts}, motion: motion{grid}} (FACE:680-709)
extern "C" int nv_element_push_motion_event(nv_element *e)
{
    nv_event_field f[2] = {{"timestamp", 1, nullptr, {0, 0, 0, 0}}, {"motion", 1, nullptr, {0, 0, 0, 0}}};
    return nv_element_push_message(e, f, 2);
}

extern "C" int nv_element_transform_frame_ip(nv_element *e, uint8_t *frame, int width, int height, int stride_bytes,
                                             uint64_t pts_ns, double now_ms)
{
    if (!e || !frame || width <= 0 || height <= 0) { nv_set_error("bad argument"); return NV_ERR_ARG; }
    int cn = e->kind == K_TRACKER ? 4 : 3;
    if (stride_bytes < width * cn) { nv_set_error("stride smaller than a row"); return NV_ERR_ARG; }
    if (!e->ctx || width > e->ctx->max_w || height > e->ctx->max_h) {       // first buffer / caps renegotiation
        nv_ctx_destroy(e->ctx); e->ctx = nullptr;
        int rc = nv_ctx_create(e->gpu, std::max(width, 1920), std::max(height, 1080), &e->ctx);
        if (rc != NV_OK) return rc;
    }
    NV_CUDA(cudaSetDevice(e->ctx->gpu));
    e->msg.clear(); e->signal.clear(); e->emitted = false; e->pushed = false;
    switch (e->kind) {
    case K_FACE: return face_frame(e, frame, width, height, stride_bytes, now_ms);
    case K_EYE: return eye_frame(e, frame, width, height, stride_bytes, now_ms);
    case K_MOUTH:
    case K_NOSE: return mouth_nose_frame(e, frame, width, height, stride_bytes, now_ms);
    case K_EAR: return ear_frame(e, frame, width, height, stride_bytes, now_ms);
    case K_TRACKER: return tracker_frame(e, frame, width, height, stride_bytes, pts_ns, now_ms);
    }
    return NV_ERR_ARG;
}

// The same call for a BGR / BGRA frame that lives in DEVICE memory (decoded and converted on the GPU, never mapped to the
// host): the frame is read where it is, and the view-* / set_visual_mode overlays are written into it by k_draw_spans —
// pixel for pixel what nv_element_transform_frame_ip draws into a host frame.  Returns after the element's stream is idle.
extern "C" int nv_element_transform_frame_device(nv_element *e, uint8_t *d_frame, int width, int height, int stride_bytes,
                                                 uint64_t pts_ns, double now_ms)
{
    if (!e || !d_frame) { nv_set_error("bad argument"); return NV_ERR_ARG; }
    const cudaMemoryType type = nv_memory_type(d_frame);
    if (type != cudaMemoryTypeDevice && type != cudaMemoryTypeManaged) {
        nv_set_error("nv_element_transform_frame_device: the frame is not in device memory");
        return NV_ERR_ARG;
    }
    e->spans.clear();
    g_span_sink = &e->spans;
    int rc = nv_element_transform_frame_ip(e, d_frame, width, height, stride_bytes, pts_ns, now_ms);
    g_span_sink = nullptr;
    if (rc != NV_OK) return rc;
    if (!e->spans.empty()) {
        rc = draw_spans_device(e->spans, d_frame, stride_bytes, e->kind == K_TRACKER ? 4 : 3, &e->d_spans, &e->d_spans_cap, e->ctx->stream);
        if (rc != NV_OK) return rc;
        e->ctx->launches++;
    }
    NV_CUDA(cudaStreamSynchronize(e->ctx->stream));
    return NV_OK;
}

static int record_shapes(uint8_t *frame, int width, int height, int stride_bytes, int channels, const nv_shape *shapes, int n,
                         std::vector<DrawSpan> &spans)
{
    g_span_sink = &spans;
    for (int i = 0; i < n; i++) {
        const nv_shape &s = shapes[i];
        const Bgr c = {s.blue, s.green, s.red};
        if (s.kind == 0) draw_rectangle3(frame, width, height, stride_bytes, channels, s.a, s.b, s.c, s.d, c);
        else if (s.kind == 1 && s.d > 1 && s.c >= 0) cvdraw::circle(frame, width, height, stride_bytes, channels, s.a, s.b, s.c, c, s.d);
        else { g_span_sink = nullptr; nv_set_error("shape %d: unknown kind or bad circle", i); return NV_ERR_ARG; }
    }
    g_span_sink = nullptr;
    return NV_OK;
}

// CPU tap of the device overlay's host half: the shapes rasterised into spans, the spans made disjoint (resolve_spans),
// then written into a HOST frame — must equal drawing the shapes one after the other (tests/test_elements_cpu.py).
extern "C" int nv_debug_draw_shapes_spans(uint8_t *frame, int width, int height, int stride_bytes, int channels,
                                          const nv_shape *shapes, int n, int *nspans)
{
    if (!frame || width <= 0 || height <= 0 || (channels != 3 && channels != 4) || stride_bytes < width * channels || n < 0 ||
        (n > 0 && !shapes)) { nv_set_error("bad argument"); return NV_ERR_ARG; }
    std::vector<DrawSpan> spans, flat;
    int rc = record_shapes(frame, width, height, stride_bytes, channels, shapes, n, spans);
    if (rc != NV_OK) return rc;
    resolve_spans(spans, flat);
    for (size_t i = 0; i < flat.size(); i++)                       // disjoint: any order gives the same picture — write them backwards
        for (size_t j = i + 1; j < flat.size(); j++)
            if (flat[i].y == flat[j].y && flat[i].xa <= flat[j].xb && flat[j].xa <= flat[i].xb) { nv_set_error("spans overlap"); return NV_ERR_STATE; }
    for (size_t k = flat.size(); k-- > 0;) {
        const DrawSpan &s = flat[k];
        for (int x = s.xa; x <= s.xb; x++) {
            uint8_t *px = frame + (size_t)s.y * stride_bytes + (size_t)x * channels;
            px[0] = (uint8_t)s.bgr; px[1] = (uint8_t)(s.bgr >> 8); px[2] = (uint8_t)(s.bgr >> 16);
            if (channels == 4) px[3] = 0;
        }
    }
    if (nspans) *nspans = (int)flat.size();
    return NV_OK;
}

extern "C" int nv_draw_shapes_device(nv_ctx *ctx, uint8_t *d_frame, int width, int height, int stride_bytes, int channels,
                                     const nv_shape *shapes, int n)
{
    if (!ctx || !d_frame || width <= 0 || height <= 0 || (channels != 3 && channels != 4) || stride_bytes < width * channels || n < 0 ||
        (n > 0 && !shapes)) { nv_set_error("bad argument"); return NV_ERR_ARG; }
    const cudaMemoryType type = nv_memory_type(d_frame);
    if (type != cudaMemoryTypeDevice && type != cudaMemoryTypeManaged) {
        nv_set_error("nv_draw_shapes_device: the frame is not in device memory");
        return NV_ERR_ARG;
    }
    std::vector<DrawSpan> spans;
    int rc = record_shapes(d_frame, width, height, stride_bytes, channels, shapes, n, spans);
    if (rc != NV_OK) return rc;
    NV_CUDA(cudaSetDevice(ctx->gpu));
    DrawSpan *d_buf = nullptr;
    size_t cap = 0;
    rc = draw_spans_device(spans, d_frame, stride_bytes, channels, &d_buf, &cap, ctx->stream);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d_buf);
    if (rc != NV_OK) return rc;
    NV_CUDA(e);
    return NV_OK;
}

// Any of the six elements fed with 4:2:0 planes (a shell whose sink caps add I420 / YV12 / NV12 / NV21): same gating,
// tracking, ROI arithmetic, events and signals; the view-* overlays are ignored — the reference defines them on BGR(A)
// pixels only.
extern "C" int nv_element_transform_frame_yuv(nv_element *e, const nv_yuv_frame *f, uint64_t pts_ns, double now_ms)
{
    if (!e || !f || f->width <= 0 || f->height <= 0) { nv_set_error("bad argument"); return NV_ERR_ARG; }
    if ((f->width & 1) || (f->height & 1)) { nv_set_error("4:2:0 frame needs even width and height"); return NV_ERR_ARG; }
    if (!e->ctx || f->width > e->ctx->max_w || f->height > e->ctx->max_h) {
        nv_ctx_destroy(e->ctx); e->ctx = nullptr;
        int rc = nv_ctx_create(e->gpu, std::max(f->width, 1920), std::max(f->height, 1080), &e->ctx);
        if (rc != NV_OK) return rc;
    }
    NV_CUDA(cudaSetDevice(e->ctx->gpu));
    e->msg.clear(); e->signal.clear(); e->emitted = false; e->pushed = false;
    const int W = f->width, H = f->height;
    e->yuv = f;
    int rc = NV_ERR_ARG;
    switch (e->kind) {
    case K_FACE: rc = face_frame(e, nullptr, W, H, 0, now_ms, f); break;
    case K_EYE: rc = eye_frame(e, nullptr, W, H, 0, now_ms); break;
    case K_MOUTH:
    case K_NOSE: rc = mouth_nose_frame(e, nullptr, W, H, 0, now_ms); break;
    case K_EAR: rc = ear_frame(e, nullptr, W, H, 0, now_ms); break;
    case K_TRACKER: rc = tracker_frame(e, nullptr, W, H, 0, pts_ns, now_ms, f); break;
    }
    e->yuv = nullptr;
    return rc;
}

extern "C" int nv_element_get_message(nv_element *e, nv_meta_rect *out, int cap, int *n, int *pushed)
{
    if (!e) { nv_set_error("null argument"); return NV_ERR_ARG; }
    int m = std::min((int)e->msg.size(), cap);
    if (out && m > 0) memcpy(out, e->msg.data(), (size_t)m * sizeof(nv_meta_rect));
    if (n) *n = m;
    if (pushed) *pushed = e->pushed ? 1 : 0;
    return NV_OK;
}

// top-level shape of the downstream event: every element builds "message" with a "timestamp" = time{pts} structure
// (FACE:196-201, EYE:237-242, MOUTH:215-220, EAR:210-215) except the nose element: "noses", no timestamp (NOSE:223)
extern "C" int nv_element_get_message_info(nv_element *e, char *name16, int *has_timestamp)
{
    if (!e) { nv_set_error("null argument"); return NV_ERR_ARG; }
    if (name16) snprintf(name16, 16, "%s", e->kind == K_NOSE ? "noses" : "message");
    if (has_timestamp) *has_timestamp = e->kind == K_NOSE ? 0 : 1;
    return NV_OK;
}

extern "C" int nv_element_get_signal(nv_element *e, char *buf, int cap, int *emitted)
{
    if (!e) { nv_set_error("null argument"); return NV_ERR_ARG; }
    if (emitted) *emitted = e->emitted ? 1 : 0;
    if (buf && cap > 0) snprintf(buf, (size_t)cap, "%s", e->emitted ? e->signal.c_str() : "");
    return NV_OK;
}

extern "C" int nv_debug_draw_rectangle(uint8_t *frame, int width, int height, int stride_bytes, int channels, int x0, int y0,
                                       int x1, int y1, int b, int g, int r)
{
    if (!frame || width <= 0 || height <= 0 || (channels != 3 && channels != 4) || stride_bytes < width * channels) {
        nv_set_error("bad argument");
        return NV_ERR_ARG;
    }
    draw_rectangle3(frame, width, height, stride_bytes, channels, x0, y0, x1, y1, Bgr{(uint8_t)b, (uint8_t)g, (uint8_t)r});
    return NV_OK;
}

extern "C" int nv_debug_draw_circle(uint8_t *frame, int width, int height, int stride_bytes, int channels, int cx, int cy,
                                    int radius, int thickness, int b, int g, int r)
{
    if (!frame || width <= 0 || height <= 0 || (channels != 3 && channels != 4) || stride_bytes < width * channels ||
        thickness < 2 || thickness > 255 || radius > 16384 || abs(cx) > (1 << 20) || abs(cy) > (1 << 20)) {
        nv_set_error("bad argument");
        return NV_ERR_ARG;
    }
    cvdraw::circle(frame, width, height, stride_bytes, channels, cx, cy, radius, Bgr{(uint8_t)b, (uint8_t)g, (uint8_t)r}, thickness);
    return NV_OK;
}

extern "C" int nv_debug_track_faces(const nv_rect *prev, const int *prev_ids, int nprev, int next_id, const nv_rect *cur,
                                    int ncur, int track_threshold, int pos_threshold, int area_threshold, nv_rect *out,
                                    int *out_ids, int cap, int *n, int *next_id_out)
{
    if ((nprev > 0 && (!prev || !prev_ids)) || (ncur > 0 && !cur) || !n) { nv_set_error("bad argument"); return NV_ERR_ARG; }
    std::vector<TrackedFace> faces, cf;
    for (int i = 0; i < nprev; i++) faces.push_back({prev[i], prev_ids[i]});
    for (int i = 0; i < ncur; i++) cf.push_back({cur[i], i});
    track_faces(faces, next_id, cf, track_threshold, pos_threshold, area_threshold);
    int m = std::min((int)faces.size(), cap);
    for (int i = 0; i < m; i++) { if (out) out[i] = faces[i].r; if (out_ids) out_ids[i] = faces[i].id; }
    *n = m;
    if (next_id_out) *next_id_out = next_id;
    return NV_OK;
}

// host-logic taps (tests/test_ref_glue.py fuzzes them against the reference's own functions, oracle/_ref)
extern "C" int nv_debug_merge_eyes_current_frame(const nv_rect *face_bb, const nv_rect *eye_r, int n_eye_r, int eye_r_same, nv_rect *eyes,
                                                 int n_eyes, int scale, int eye_left, int cap, int *n)
{
    if (!face_bb || !n || n_eyes < 0 || n_eye_r < 0 || (n_eyes > 0 && !eyes) || (n_eye_r > 0 && !eye_r)) { nv_set_error("bad argument"); return NV_ERR_ARG; }
    std::vector<nv_rect> er(eye_r, eye_r + n_eye_r), ev(eyes, eyes + n_eyes);
    merge_eyes_current_frame(*face_bb, eye_r_same ? &ev : &er, ev, scale, eye_left != 0);
    int m = std::min((int)ev.size(), cap);
    for (int i = 0; i < m; i++) eyes[i] = ev[i];
    *n = (int)ev.size();
    return NV_OK;
}

extern "C" int nv_debug_merge_consecutive(int kind, const nv_rect *cur, int ncur, const nv_rect *prev, int nprev, const nv_rect *face,
                                          int scale, nv_rect *out, int cap, int *n)
{
    if (kind < 0 || kind > 2 || !face || !n || ncur < 0 || nprev < 0 || (ncur > 0 && !cur) || (nprev > 0 && !prev)) { nv_set_error("bad argument"); return NV_ERR_ARG; }
    std::vector<nv_rect> c(cur, cur + ncur), p(prev, prev + nprev);
    auto r = merge_consecutive(c, p, kind == 0 ? 7 : kind == 1 ? 4 : 6, kind != 0, *face, scale);   // DEFAULT_EUCLIDEAN_DIS: EYE:43, MOUTH:25, NOSE:43
    int m = std::min((int)r.size(), cap);
    for (int i = 0; i < m; i++) out[i] = r[i];
    *n = (int)r.size();
    return NV_OK;
}

extern "C" int nv_debug_eye_to_global(nv_rect *eyes, int n, const nv_rect *face, int scale)
{
    if (!face || n < 0 || (n > 0 && !eyes)) { nv_set_error("bad argument"); return NV_ERR_ARG; }
    std::vector<nv_rect> v(eyes, eyes + n);
    to_global(v, *face, scale);
    for (int i = 0; i < n; i++) eyes[i] = v[i];
    return NV_OK;
}

extern "C" void nv_debug_set_wall_clock_ms(double ms) { g_wall_override_ms = ms; }
