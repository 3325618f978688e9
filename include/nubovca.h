/*
 * nubovca.h — C ABI of libnubovca.so: the B200-native (sm_100a) per-frame detection hot path of
 * NUBOMEDIA-VCA.  Each entry point replaces the OpenCV call block one reference element makes
 * per video buffer; the reference file:line it stands in for is cited beside it
 * (paths relative to /root/reference/modules/<mod>/<mod-dir>/src/gst-plugins/).
 *
 * Conventions
 *   - plain C, no exceptions cross the boundary; every function returns NV_OK (0) or a negative
 *     nv_status, and nv_last_error() gives a thread-local message for the last failure.
 *   - the caller owns input frames and output arrays; the library owns all device and pinned
 *     memory inside nv_ctx.  Host input is fully consumed before a synchronous call returns
 *     (the element unmaps the GstBuffer right after, kmsfacedetect.cpp:888).
 *   - one nv_ctx per element instance (it carries the element's per-stream state: CUDA stream,
 *     scratch, tracker history).  A ctx is not thread-safe; the element shell serialises calls
 *     with its own mutex exactly as the reference does (kmsfacedetect.cpp:873-885).  Any number
 *     of contexts may run concurrently on one GPU and across GPUs.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *     NV_ERR_NO_DEVICE.
 */
#ifndef NUBOVCA_H
#define NUBOVCA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NV_API __attribute__((visibility("default")))

typedef enum {
    NV_OK = 0,
    NV_ERR_ARG = -1,          /* bad pointer / size / parameter                               */
    NV_ERR_CUDA = -2,         /* a CUDA runtime call failed (message in nv_last_error)        */
    NV_ERR_IO = -3,           /* cascade file unreadable                                      */
    NV_ERR_FORMAT = -4,       /* cascade XML malformed                                        */
    NV_ERR_UNSUPPORTED = -5,  /* cascade is neither a BOOST/HAAR nor a BOOST/LBP model (HOG)  */
    NV_ERR_CAPACITY = -6,     /* frame larger than the ctx was created for, or too many levels */
    NV_ERR_NO_DEVICE = -7,    /* no CUDA device: the library never computes on the CPU        */
    NV_ERR_STATE = -8         /* call order violated (collect without submit, ...)            */
} nv_status;

typedef struct nv_ctx nv_ctx;
typedef struct nv_cascade nv_cascade;

/* cv::Rect as the elements store it (vector<Rect>, kmsfacedetect.cpp:792) */
typedef struct { int x, y, width, height; } nv_rect;

NV_API const char *nv_version(void);
NV_API const char *nv_last_error(void);
NV_API int nv_device_count(void);                       /* 0 when no CUDA device is visible */

/* ---- cascade model: replaces cv::CascadeClassifier::load (kmsfacedetect.cpp:163-177,
 *      kmseyedetect.cpp:171-183, kmsmouthdetect.cpp:157-163, kmsnosedetect.cpp:166-172,
 *      kmseardetect.cpp:173-186).  Host-side parse only; usable without a GPU.  BOOST/HAAR cascades in
 *      the new or the OpenCV 1.x/2.x XML layout: stumps or trees, upright or tilted features; BOOST/LBP
 *      cascades (new layout; categorical stumps or trees over the 256 LBP codes, SURVEY §8f rank 3). -- */
typedef struct {
    int win_w, win_h;        /* training window                                   */
    int nstages, nstumps;    /* boosted stages / weak classifiers (stumps)        */
    int nfeatures;           /* Haar features (<= 3 rects each)                   */
    int n3rect;              /* features that use the third rectangle             */
    int order_free_sums;     /* 1: every stage sum is exact in double in any order */
    int general;             /* 1: trees of more than one node and/or tilted features (OpenCV's predictOrdered path) */
    int has_tilted;          /* 1: some feature is evaluated on the tilted integral */
    int nnodes;              /* internal tree nodes over all weak classifiers (== nstumps for stump cascades) */
    int lbp;                 /* 1: LBP features (OpenCV's predictCategorical path; no variance normalisation) */
} nv_cascade_info;

NV_API int nv_cascade_load(const char *xml_path, nv_cascade **out);
NV_API int nv_cascade_get_info(const nv_cascade *c, nv_cascade_info *info);
NV_API void nv_cascade_free(nv_cascade *c);

/* ---- context ------------------------------------------------------------------------------ */
NV_API int nv_ctx_create(int gpu, int max_width, int max_height, nv_ctx **out);
NV_API void nv_ctx_destroy(nv_ctx *ctx);
/* debug != 0 makes the cascade kernels also write per-window stage-exit depth maps
 * (same kernels, same arithmetic — a template flag adds the stores). */
NV_API int nv_ctx_set_debug(nv_ctx *ctx, int debug);

/* ---- CascadeClassifier::detectMultiScale on an 8-bit gray image
 *      (kmsfacedetect.cpp:809-811, kmseyedetect.cpp:958-960,991-993,1003-1005,
 *       kmsmouthdetect.cpp:845-848,870-873, kmsnosedetect.cpp:843-846,870-873,
 *       kmseardetect.cpp:656-659,712-715).  `flags` is accepted and ignored, as OpenCV >= 3
 *      ignores it for new-format cascades.  max_w/max_h == 0 means "image size". ---------------- */
typedef struct {
    double scale_factor;
    int min_neighbors;
    int flags;
    int min_w, min_h;
    int max_w, max_h;
} nv_detect_params;

NV_API int nv_detect_multiscale(nv_ctx *ctx, const nv_cascade *c, const uint8_t *gray, int width, int height,
                                int stride_bytes, const nv_detect_params *p, nv_rect *out, int cap, int *n);

/* ---- detection scores: cv::CascadeClassifier::detectMultiScale2 / detectMultiScale3 (OpenCV 4.13).
 *      on != 0: every detect call on this ctx (nv_detect_multiscale, nv_face_detect / _submit / _submit_device /
 *      _detect_yuv / _submit_yuv) also yields, per output rectangle, detectMultiScale2's numDetections and
 *      detectMultiScale3(outputRejectLevels = true)'s levelWeights:
 *        - min_neighbors > 0: numDetections is the number of raw windows grouped into the rectangle (the count compared
 *          with min_neighbors), levelWeight the largest last-stage sum among them;
 *        - min_neighbors <= 0: numDetections is 1, levelWeight the window's own last-stage sum.
 *      A window's last-stage sum is the double sum of its last stage's leaves in XML order, which is at or above that
 *      stage's threshold.  detectMultiScale3's rejectLevels is always the cascade's stage count and is not returned.
 *      The setting applies from the next submit; a ctx keeps separate graphs for both settings.  Rectangles do not change. */
NV_API int nv_ctx_set_scores(nv_ctx *ctx, int on);
/* Scores of the last collected call, parallel to its rectangles (same order, same clip); either output may be NULL.
 * NV_ERR_STATE if that call ran with scores off; NV_ERR_CAPACITY (and the first cap entries) if cap is too small. */
NV_API int nv_get_scores(nv_ctx *ctx, int *neighbors, double *level_weights, int cap, int *n);

/* ---- the nubofacedetector hot block, kmsfacedetect.cpp:770-811:
 *      scale = width / width_to_process (integer), cv::resize(BGR, INTER_LINEAR), BGR2GRAY,
 *      equalizeHist, detectMultiScale(scale_factor, min_neighbors, 0, Size(min_w, min_h)).
 *      min_w < 0 selects the element's own rule Size(cols/20, rows/20) (:811).
 *      Rectangles are in processing-size coordinates, like the reference's current_faces. ------ */
typedef struct {
    int width_to_process;
    double scale_factor;      /* MULTI_SCALE_FACTOR(prop) = 1 + prop/100, kmsfacedetect.cpp:142 */
    int min_neighbors;        /* 3 in the reference                                            */
    int min_w, min_h;
} nv_face_params;

NV_API int nv_face_detect(nv_ctx *ctx, const nv_cascade *c, const uint8_t *bgr, int width, int height,
                          int stride_bytes, const nv_face_params *p, nv_rect *out, int cap, int *n);

/* Asynchronous halves of nv_face_detect, so that one host thread can keep many per-stream
 * contexts in flight (BASELINE config 5: 32 streams per GPU).  submit() enqueues copy + kernels on the
 * ctx's CUDA stream; collect() waits for that stream and returns the rectangles.  A pageable frame is
 * first copied into the ctx's pinned staging buffer (the caller may reuse it as soon as submit returns); a
 * frame in page-locked memory (cudaHostAlloc / cudaHostRegister) is read directly by the DMA engine and
 * must stay untouched until collect.  Once a context sees the same call shape twice, the whole per-frame
 * kernel sequence is replayed as a single CUDA graph launch.  When width / width_to_process is 3 or more and divides
 * both dimensions, cv::resize(INTER_LINEAR) reads only two of every `scale` source rows: only those rows are read from
 * the caller's frame and copied to the device (half of a 640x480 frame processed at 160x120). */
NV_API int nv_face_submit(nv_ctx *ctx, const nv_cascade *c, const uint8_t *bgr, int width, int height,
                          int stride_bytes, const nv_face_params *p);
NV_API int nv_face_collect(nv_ctx *ctx, nv_rect *out, int cap, int *n);

/* Same pipeline with the frame already resident in device memory (bench.py `value`: inputs in
 * HBM when the timed region starts).  d_bgr must stay valid until collect. */
NV_API int nv_face_submit_device(nv_ctx *ctx, const nv_cascade *c, const uint8_t *d_bgr, int width, int height,
                                 int stride_bytes, const nv_face_params *p);

/* Page-locked host memory for frames (what a GstAllocator / buffer pool of the shell hands upstream, so that
 * decoded frames land where the DMA engine reads them without a staging copy).  Portable across devices. */
NV_API int nv_host_alloc(size_t bytes, void **out);
NV_API void nv_host_free(void *p);
/* Page-lock memory the caller already owns (cudaHostRegister, portable): what a shell does once per block of the upstream
 * buffer pool when it cannot hand out nv_host_alloc memory.  Frames inside a registered block take the no-staging path. */
NV_API int nv_host_register(void *p, size_t bytes);
NV_API int nv_host_unregister(void *p);

/* ---- batches: N images of one size per call, through one chain of kernel launches ---------------------------------------
 *      frames: N pointers to N images (8-bit gray for nv_detect_multiscale_batch, BGR for the face calls), each `height`
 *      rows of `stride_bytes`.  on_device == 0: host memory, copied like the single calls' frames (page-locked frames are
 *      read by the DMA engine in place and must stay untouched until collect, pageable ones are staged before submit
 *      returns; for the face calls only the row pairs the resize reads travel, as in nv_face_submit).  on_device != 0:
 *      device pointers (a CUDA uint8 tensor [N, H, W(, 3)]: data_ptr() + i * stride(0)), read in place until collect.
 *      Image i's rectangles are exactly those of the single call on that image (nv_detect_multiscale / nv_face_detect,
 *      same nv_face_params rules, min_w < 0 included).  out holds image 0's rectangles, then image 1's, ...; counts[i] is
 *      always image i's true count and *total (if given) the number written; when the counts add up to more than cap, the
 *      first cap rectangles are written and the call returns NV_ERR_CAPACITY.
 *      Route: when the image size makes a small plan (at most 16384 windows) of a stump cascade with the order-free
 *      exactness certificates whose weak classifiers fit in shared memory (haarcascade_frontalface_alt on a 160x120 or
 *      96x64 image: the face element's default shape), the whole batch runs as ONE chain of six kernel launches (five for
 *      gray images), replayed as one CUDA graph once the shape (N, size, cascade, parameters) repeats — new frame addresses
 *      on every call do not prevent the replay.  An image with more than 1024 raw candidates is detected again alone in
 *      collect.  Every other case (larger images, tree / tilted / LBP models, models without the certificates) runs the
 *      single-image pipeline once per image inside submit: the same results, no gain in throughput.
 *      The context grows its per-image buffers to the largest batch it has seen and keeps them.  A batch shares the
 *      context's cache of plans with the single calls: a batch shape that is not cached takes the least recently used
 *      plan (and that plan's single-call graph) and may grow the single-call integral buffers, so a single call after it
 *      can re-plan once; results never depend on it.
 *      Refused: N < 1 or N > NV_BATCH_MAX (NV_ERR_ARG); a context with scores on (NV_ERR_STATE).  After a batch,
 *      nv_debug_get_counters reports [0..2] summed over its images, [3] the kernel launches of the whole call and [4] 1 when
 *      the batched chain was replayed from a CUDA graph captured by an earlier call (0 otherwise); the other
 *      parity taps, nv_get_scores and nv_ctx_get_stage_times return NV_ERR_STATE (they describe single calls); a pending
 *      batch is collected with nv_face_collect_batch only.  Batches of 4:2:0 frames: nv_face_submit_batch_yuv /
 *      nv_face_detect_batch_yuv below. ------------------------------------------------------------------------------------ */
#define NV_BATCH_MAX 256
NV_API int nv_detect_multiscale_batch(nv_ctx *ctx, const nv_cascade *c, const uint8_t *const *frames, int n, int width, int height,
                                      int stride_bytes, int on_device, const nv_detect_params *p, nv_rect *out, int cap, int *counts);
NV_API int nv_face_submit_batch(nv_ctx *ctx, const nv_cascade *c, const uint8_t *const *frames, int n, int width, int height,
                                int stride_bytes, int on_device, const nv_face_params *p);
NV_API int nv_face_collect_batch(nv_ctx *ctx, nv_rect *out, int cap, int *counts, int *total);
NV_API int nv_face_detect_batch(nv_ctx *ctx, const nv_cascade *c, const uint8_t *const *frames, int n, int width, int height,
                                int stride_bytes, int on_device, const nv_face_params *p, nv_rect *out, int cap, int *counts,
                                int *total);

/* ---- 4:2:0 ingest (extension, SURVEY §8f rank 4).  The reference elements negotiate BGR only
 *      (kmsfacedetect.cpp:129-133,1025-1031), so a decoder's I420 / NV12 output passes through a CPU videoconvert
 *      and twice the bytes cross PCIe.  These entry points take the decoder's planes as they are: the result is
 *      what nv_face_detect gives on cv::cvtColor(frame, COLOR_YUV2BGR_I420 / _NV12 / _NV21) — the conversion is
 *      applied per source pixel inside the resize + gray kernel (BT.601, OpenCV's 20-bit fixed point), the BGR
 *      frame never exists.  YV12 is I420 with plane[1] and plane[2] swapped by the caller.  width and height even.
 *      plane[2] / stride[2] are ignored for NV12 / NV21.  on_device != 0: the planes are device pointers.
 *      The planes need not share an allocation: they travel as one copy only when they follow each other with at most a
 *      row of padding in between, otherwise plane by plane (each plane's own page-lock state is honoured). ------------- */
typedef enum { NV_FMT_BGR = 0, NV_FMT_I420 = 1, NV_FMT_NV12 = 2, NV_FMT_NV21 = 3 } nv_pixel_format;
typedef struct {
    int format;               /* nv_pixel_format, one of the 4:2:0 values */
    int width, height;
    const uint8_t *plane[3];
    int stride[3];
    int on_device;
} nv_yuv_frame;

NV_API int nv_face_detect_yuv(nv_ctx *ctx, const nv_cascade *c, const nv_yuv_frame *f, const nv_face_params *p,
                              nv_rect *out, int cap, int *n);
NV_API int nv_face_submit_yuv(nv_ctx *ctx, const nv_cascade *c, const nv_yuv_frame *f, const nv_face_params *p);   /* + nv_face_collect */
/* Batches of 4:2:0 frames: the face batch calls above (same route, results, counts, capacity, limits and refusals; a pending
 * batch is collected with nv_face_collect_batch) on n decoder frames.  Every frame passes the checks of nv_face_detect_yuv,
 * and all share format, width, height, plane strides (stride[2] of I420 only) and on_device, else NV_ERR_ARG naming the
 * first frame that differs.  Each frame's planes may lie anywhere: one block or scattered, pageable, page-locked (read in
 * place until collect) or, with on_device, device memory (read in place, no copy).  Image i's rectangles are exactly
 * those of nv_face_detect_yuv on frame i.  On the batched route, host frames travel plane by plane: of the luma plane only
 * the row pairs the resize reads, the chroma planes whole.  A 640x480 NV12 frame processed at 160x120 moves 307 200 bytes
 * (120 luma row pairs, 153 600 bytes, and the 153 600-byte chroma plane), against 460 800 for the BGR frame's row pairs in
 * nv_face_detect_batch. */
NV_API int nv_face_submit_batch_yuv(nv_ctx *ctx, const nv_cascade *c, const nv_yuv_frame *frames, int n,
                                    const nv_face_params *p);
NV_API int nv_face_detect_batch_yuv(nv_ctx *ctx, const nv_cascade *c, const nv_yuv_frame *frames, int n,
                                    const nv_face_params *p, nv_rect *out, int cap, int *counts, int *total);
/* cvtColor(COLOR_YUV2BGR_*) alone, host in / host out (parity tap of the ingest arithmetic) */
NV_API int nv_yuv2bgr(nv_ctx *ctx, const nv_yuv_frame *f, uint8_t *dst_bgr, int dst_stride);

/* ---- the nubotracker per-frame block, gstnubotracker.cpp:356-380: BGRA->gray, absdiff with the
 *      previous frame, threshold, updateMotionHistory(ts, 0.2), segmentMotion(ts, 32),
 *      __join_objects.  The reference's timestamp is clock() in ms (:349); it is injected here.
 *      The first frame after create only primes the history (num_frames == 0, :360). ---------- */
typedef struct {
    int threshold;            /* set_threshold, default 20    */
    int min_area;             /* set_min_area, default 50     */
    long max_area;            /* set_max_area, default 30000  */
    int distance;             /* set_distance, default 35     */
} nv_tracker_params;

NV_API int nv_tracker_process(nv_ctx *ctx, const uint8_t *bgra, int width, int height, int stride_bytes,
                              double timestamp_ms, const nv_tracker_params *p, nv_rect *out, int cap, int *n);
NV_API int nv_tracker_reset(nv_ctx *ctx);
/* The same block fed with 4:2:0 planes (ingest extension, see nv_face_detect_yuv): gray is BGR2GRAY of
 * cvtColor(COLOR_YUV2BGR_*) per pixel, i.e. the result equals nv_tracker_process on the converted frame. */
NV_API int nv_tracker_process_yuv(nv_ctx *ctx, const nv_yuv_frame *frame, double timestamp_ms, const nv_tracker_params *p,
                                  nv_rect *out, int cap, int *n);
/* Batched tracker: many video streams on one context, one kernel launch and one synchronise per call.  The context keeps up
 * to NV_BATCH_MAX stream slots, each with its own tracker state; frame i of a call is the next frame of slot i, with
 * timestamps_ms[i] and params[i] (streams may differ in threshold, areas and distance).  Slot i's rectangles are exactly
 * those nv_tracker_process / nv_tracker_process_yuv give on a separate context fed slot i's frames, timestamps and
 * parameters.
 *   Frames: BGRA, height rows of stride_bytes (a multiple of 4), or 4:2:0 frames that all share format, size, plane strides
 *   and on_device (else NV_ERR_ARG naming the first frame that differs); each frame passes the single call's checks.
 *   Pageable, page-locked (read in place by the copy engine) or, with on_device, device memory (read in place, no copy;
 *   a CUDA uint8 tensor [N, H, W, 4]: data_ptr() + i * stride(0), at any byte address).
 *   Output as in nv_face_detect_batch: out holds image 0's rectangles, then image 1's, ...; counts[i] is always image i's
 *   count after __join_objects, *total (if given) the number written; more than cap in all: the first cap are written and
 *   the call returns NV_ERR_CAPACITY.  An image with more than 16384 raw motion components gets the single call's truncated
 *   result and the call returns NV_ERR_CAPACITY naming it, after every image has been written.
 *   More than 255 distinct timestamps inside a slot's 0.2 ms motion-history window: NV_ERR_CAPACITY naming the slot, checked
 *   for every slot before anything runs, so no slot changes.  Refused with NV_ERR_ARG: n outside 1 .. NV_BATCH_MAX, a null
 *   table, timestamps, params or counts (out may be null with cap 0); a frame larger than the context: NV_ERR_CAPACITY, as
 *   in the single call.
 *   Slots: a slot's first frame after creation, reset or reconfiguration only primes it (0 rectangles).  The slots grow to the
 *   largest n seen; a call with a smaller n leaves the higher slots as they are, to continue later.  All slots share one
 *   frame size: a call at another size starts every slot afresh.  The slots share nothing with nv_tracker_process, and a
 *   tracker batch leaves a pending nv_face_submit* / nv_face_submit_batch* as it is.  With profiling on,
 *   nv_ctx_get_tracker_kernel_ms reports the batched kernel of the last call.  Blocking, like nv_tracker_process. */
NV_API int nv_tracker_process_batch(nv_ctx *ctx, const uint8_t *const *frames, int n, int width, int height, int stride_bytes,
                                    int on_device, const double *timestamps_ms, const nv_tracker_params *params, nv_rect *out,
                                    int cap, int *counts, int *total);
NV_API int nv_tracker_process_batch_yuv(nv_ctx *ctx, const nv_yuv_frame *frames, int n, const double *timestamps_ms,
                                        const nv_tracker_params *params, nv_rect *out, int cap, int *counts, int *total);
NV_API int nv_tracker_reset_batch(nv_ctx *ctx, int slot);   /* clears one slot; slot < 0: every slot */

/* ---- image ops used by the nested elements (eye/mouth/nose/ear) on host images:
 *      cvtColor BGR2GRAY (kmseyedetect.cpp:949), equalizeHist (:950,964), cv::resize INTER_LINEAR
 *      (:956,963), cv::flip(…,1) (kmseardetect.cpp:800). ------------------------------------- */
NV_API int nv_bgr2gray(nv_ctx *ctx, const uint8_t *src, int width, int height, int stride_bytes, int channels,
                       uint8_t *dst_gray, int dst_stride);
NV_API int nv_equalize_hist(nv_ctx *ctx, const uint8_t *src, int width, int height, int stride_bytes,
                            uint8_t *dst, int dst_stride);
NV_API int nv_resize_linear(nv_ctx *ctx, const uint8_t *src, int width, int height, int stride_bytes, int channels,
                            uint8_t *dst, int dst_width, int dst_height, int dst_stride);
NV_API int nv_flip_horizontal(nv_ctx *ctx, const uint8_t *src, int width, int height, int stride_bytes,
                              uint8_t *dst, int dst_stride);

/* ---- element mirrors: the per-frame logic of the six GStreamer elements without GStreamer.
 *      Same factory names (kmsfacedetect.cpp:21, kmseyedetect.cpp:23, kmsmouthdetect.cpp:19,
 *      kmsnosedetect.cpp:24, kmseardetect.cpp:24, gstnubotracker.cpp:22), same GObject property names,
 *      ranges and defaults (kmsfacedetect.cpp:1043-1102, kmseyedetect.cpp:1274-1320, kmsmouthdetect.cpp:
 *      1078-1121, kmsnosedetect.cpp:1090-1133, kmseardetect.cpp:995-1038, gstnubotracker.cpp:504-542),
 *      same frame gating, ROI arithmetic, temporal smoothing, downstream "message" structures and
 *      signal strings.  A GStreamer shell only has to forward properties, sink events and buffers
 *      (INTEGRATION.md).  nv_element_transform_frame_ip stands in for GstVideoFilterClass::
 *      transform_frame_ip (kmsfacedetect.cpp:857-898, kmseyedetect.cpp:1107-1141,
 *      kmsmouthdetect.cpp:912-946, kmsnosedetect.cpp:915-955, kmseardetect.cpp:830-866,
 *      gstnubotracker.cpp:423-445); it always succeeds from the pipeline's point of view
 *      (the reference always returns GST_FLOW_OK): failures are reported through the return code and
 *      the frame passes through untouched. ------------------------------------------------------- */
typedef struct nv_element nv_element;

/* one sub-structure of the downstream custom event ("message"/"noses" GstStructure) */
typedef struct {
    char name[16];            /* structure name: "face", "eye_left", "eye_right", "mouth", "noses", "face_profile", "ear" */
    char type[16];            /* its "type" field: "face", "eye", "mouth", "nose", "face_profile", "ear"               */
    unsigned x, y, width, height;
} nv_meta_rect;

/* cascade_dir: where the haarcascade_*.xml models live (NULL: $NUBOVCA_CASCADE_DIR, else /usr/share/opencv/haarcascades, the
 * reference's hard-coded directory).  A model that cannot be loaded is not fatal, as in the reference (kmsfacedetect.cpp:
 * 167-171): the call returns NV_OK and nv_last_error() holds a "warning: ..." text naming the files (empty otherwise).
 * Known behavioural difference: the reference passes CV_HAAR_FIND_BIGGEST_OBJECT to the mouth / nose / ear ROI cascades;
 * with the OpenCV 2.x it linked and OLD-format models that flag keeps at most one object per ROI, while OpenCV >= 3 (the
 * oracle of this library, cv2 4.13) ignores `flags` for new-format models and returns every grouped rectangle — and so
 * does this library. */
NV_API int nv_element_create(const char *factory_name, int gpu, const char *cascade_dir, nv_element **out);
NV_API void nv_element_destroy(nv_element *e);
NV_API int nv_element_set_property(nv_element *e, const char *name, long value);
NV_API int nv_element_get_property(nv_element *e, const char *name, long *value);
/* property table of the element, for a shell that installs its GObject properties from it (kmsfacedetect.cpp:1043-1102
 * and the analogous class_init blocks): index 0 .. count-1; returns NV_ERR_ARG past the end.  *name stays valid for
 * the element's lifetime. */
NV_API int nv_element_property_info(nv_element *e, int index, const char **name, long *minimum, long *maximum, long *default_value);
/* sink_event: a queued upstream "message" carrying face rectangles (kmseyedetect.cpp:192-218,680-724),
 * or the "motion" event the face element waits for in detect-event mode (kmsfacedetect.cpp:698-707) */
/* General form: one custom downstream event as the element's sink pad saw it, field by field.  The reference queues a copy of
 * EVERY such event (kmsfacedetect.cpp:258-267, kmseyedetect.cpp:198-209) and __receive_event pops exactly one per frame,
 * whatever it holds (kmsfacedetect.cpp:711-755, kmseyedetect.cpp:726-764): a message without a structure-typed "timestamp"
 * field is dropped unread; the face element re-arms only on a structure-typed "motion" field; eye and nose keep the
 * sub-structures whose "type" is "face" and accept the message if it holds any structure field (kmseyedetect.cpp:680-724,
 * kmsnosedetect.cpp:648-694); the mouth element only looks at fields named "0", "1", ... in that order
 * (kmsmouthdetect.cpp:655-703).  The ear element and the tracker have no sink_event handler. */
typedef struct {
    const char *name;         /* field name in the message: "timestamp", "0", "1", "motion", ...                 */
    int is_structure;         /* the field holds a GstStructure                                                   */
    const char *type;         /* that structure's "type" string; NULL if it has none                              */
    nv_rect rect;             /* its x / y / width / height (G_TYPE_UINT fields; 0 where absent)                  */
} nv_event_field;
NV_API int nv_element_push_message(nv_element *e, const nv_event_field *fields, int nfields);
/* shorthands: a face message {timestamp, faces...} / a motion message {timestamp, motion} */
NV_API int nv_element_push_faces_event(nv_element *e, const nv_rect *faces, int n);
NV_API int nv_element_push_motion_event(nv_element *e);
/* one video buffer.  frame: BGR (detectors) or BGRA (tracker), modified in place only when a view-*
 * property asks for it (cvRectangle / cv::circle restated pixel-exactly, see nv_debug_draw_*).  now_ms < 0 uses gettimeofday for
 * the events-ms rate limit.  The tracker's motion-history timestamp is pts_ns / 1e6 ms (the reference uses clock(), the
 * process's CPU time, gstnubotracker.cpp:349 — not a media clock; deliberate deviation). */
NV_API int nv_element_transform_frame_ip(nv_element *e, uint8_t *frame, int width, int height, int stride_bytes,
                                         uint64_t pts_ns, double now_ms);
/* The same for a BGR / BGRA frame in DEVICE memory (SURVEY §8f rank 4: frames decoded and converted on the GPU): read in
 * place, overlays written by a kernel — the same pixels nv_element_transform_frame_ip writes into a host frame. */
NV_API int nv_element_transform_frame_device(nv_element *e, uint8_t *d_frame, int width, int height, int stride_bytes,
                                             uint64_t pts_ns, double now_ms);
/* cvRectangle(.., thickness 3, 8, 0) / cv::circle(.., thickness, 8, 0) into a BGR(A) frame in device memory, on the ctx's
 * stream (returns after it is idle): shapes are drawn in array order, the later one wins where they overlap.
 * kind 0: rectangle with corners (a, b) .. (c, d); kind 1: circle with centre (a, b), radius c, thickness d (> 1). */
typedef struct { int kind, a, b, c, d; unsigned char blue, green, red, pad; } nv_shape;
NV_API int nv_draw_shapes_device(nv_ctx *ctx, uint8_t *d_frame, int width, int height, int stride_bytes, int channels,
                                 const nv_shape *shapes, int n);
/* Any of the six elements on 4:2:0 planes (see nv_face_detect_yuv / nv_tracker_process_yuv; the nested elements take
 * their full-resolution gray image as BGR2GRAY(cvtColor(COLOR_YUV2BGR_*)) per pixel): gating, tracking, ROI arithmetic,
 * events and signals as above; the view-* / set_visual_mode overlays are ignored (the reference defines them on BGR(A)
 * pixels). */
NV_API int nv_element_transform_frame_yuv(nv_element *e, const nv_yuv_frame *frame, uint64_t pts_ns, double now_ms);
/* what the last frame produced: the downstream event's sub-structures (pushed != 0 if the element
 * pushed the event; the ear element builds it but never pushes, kmseardetect.cpp:210-290) and the
 * signal payload ("x:..,y:..,width:..,height:..;" repeated) if the signal fired */
NV_API int nv_element_get_message(nv_element *e, nv_meta_rect *out, int cap, int *n, int *pushed);
NV_API int nv_element_get_signal(nv_element *e, char *buf, int cap, int *emitted);
/* top-level shape of that event: structure name ("message"; "noses" for the nose element, kmsnosedetect.cpp:223) and whether
 * it starts with timestamp = time{pts} (every element but the nose one); sub-structure i is set under field name "i" */
NV_API int nv_element_get_message_info(nv_element *e, char *name16, int *has_timestamp);
/* host-logic taps for unit tests: Faces::track_faces (Faces.cpp:78-153) on explicit lists */
/* cvRectangle(img, (x0, y0), (x1, y1), Scalar(b, g, r, 0), 3, 8, 0) on a 3- or 4-channel host frame: the drawing the
 * view-faces / view-mouths / view-noses / view-ears properties and the tracker's visual mode perform in place
 * (BaseFace.cpp:76, kmsmouthdetect.cpp:900, kmsnosedetect.cpp:902, kmseardetect.cpp:754, gstnubotracker.cpp:389). */
NV_API int nv_debug_draw_rectangle(uint8_t *frame, int width, int height, int stride_bytes, int channels, int x0, int y0,
                                   int x1, int y1, int b, int g, int r);
/* cv::circle(img, (cx, cy), radius, Scalar(b, g, r, 0), thickness >= 2, 8, 0): the view-eyes drawing
 * (kmseyedetect.cpp:1081,1095 use thickness 4). */
/* the host half of nv_draw_shapes_device on a HOST frame: shapes -> spans -> disjoint spans -> pixels (CPU test tap) */
NV_API int nv_debug_draw_shapes_spans(uint8_t *frame, int width, int height, int stride_bytes, int channels,
                                      const nv_shape *shapes, int n, int *nspans);
NV_API int nv_debug_draw_circle(uint8_t *frame, int width, int height, int stride_bytes, int channels, int cx, int cy,
                                int radius, int thickness, int b, int g, int r);
/* tests: replace gettimeofday() in the events-ms rate limit and the activate-events setter (kmsfacedetect.cpp:228-236,
 * 556-560) by a fixed value; negative restores the real clock.  Process-wide. */
NV_API void nv_debug_set_wall_clock_ms(double ms);
NV_API int nv_debug_track_faces(const nv_rect *prev, const int *prev_ids, int nprev, int next_id, const nv_rect *cur,
                                int ncur, int track_threshold, int pos_threshold, int area_threshold, nv_rect *out,
                                int *out_ids, int cap, int *n, int *next_id_out);
/* __merge_eyes_current_frame (kmseyedetect.cpp:778-862), in place on `eyes` (*n = resulting count); eye_r_same != 0 is the
 * right eye's call shape, where the eye_r argument IS the list being merged (kmseyedetect.cpp:1016) */
NV_API int nv_debug_merge_eyes_current_frame(const nv_rect *face_bb, const nv_rect *eye_r, int n_eye_r, int eye_r_same, nv_rect *eyes,
                                             int n_eyes, int scale, int eye_left, int cap, int *n);
/* kind 0: __merge_eyes_consecutives_frames (kmseyedetect.cpp:864-900), 1: __merge_mouths_consecutives_frames
 * (kmsmouthdetect.cpp:750-796), 2: __merge_noses_consecutives_frames (kmsnosedetect.cpp:745-790) */
NV_API int nv_debug_merge_consecutive(int kind, const nv_rect *cur, int ncur, const nv_rect *prev, int nprev, const nv_rect *face,
                                      int scale, nv_rect *out, int cap, int *n);
/* transform_2_global_coordinates (kmseyedetect.cpp:902-913), in place */
NV_API int nv_debug_eye_to_global(nv_rect *eyes, int n, const nv_rect *face, int scale);
/* __join_objects / __merge / calc_dist (gstnubotracker.cpp:119-200), in place (*n = resulting count) */
NV_API int nv_debug_join_objects(nv_rect *rects, int n_in, int min_area, long max_area, int distance, int *n);

/* ---- device-side timing (bench.py): CUDA events on the ctx's own stream.  With profiling on, every
 *      pipeline stage of a detect call is bracketed by events; times are read after collect.
 *      Stage slots: see nv_stage_name(). ------------------------------------------------------ */
#define NV_NUM_STAGES 8
NV_API const char *nv_stage_name(int slot);
NV_API int nv_ctx_set_profile(nv_ctx *ctx, int on);
NV_API int nv_ctx_get_stage_times(nv_ctx *ctx, float *ms, int cap, int *n);   /* last collected call */
NV_API int nv_ctx_get_tracker_kernel_ms(nv_ctx *ctx, float *ms);              /* the fused kernel of the last nv_tracker_process */
NV_API int nv_event_create(void **ev);
NV_API int nv_event_record(nv_ctx *ctx, void *ev);                             /* on the ctx's stream */
NV_API int nv_event_elapsed_ms(void *ev_start, void *ev_end, float *ms);       /* waits for ev_end   */
NV_API void nv_event_destroy(void *ev);

/* ---- parity taps (tests only): artefacts of the LAST detect call on this ctx ---------------- */
typedef struct {
    float scale;
    int width, height;        /* level image size                                   */
    int ystep;
    int nx, ny;               /* window grid actually visited (x and y in ystep units) */
} nv_level_info;

#define NV_DEPTH_PASS 1
#define NV_DEPTH_VARREJ (-100)     /* OpenCV result -1 from the variance test                 */
#define NV_DEPTH_SKIPPED (-32768)  /* never evaluated: stage-0 skip rule                      */
/* other values: 0 = failed stage 0, -k = failed stage k                                       */

/* model taps: what the XML loader produced (cross-checked against an independent parser in tests) */
NV_API int nv_debug_cascade_stage(const nv_cascade *c, int stage, int *ntrees, float *threshold_used);
NV_API int nv_debug_cascade_stump(const nv_cascade *c, int stump, int rects12[12], float weights3[3],
                                  float thr_left_right[3]);
/* weak classifier `tree` of any cascade: internal nodes in file order (feature index, child on "<", child otherwise;
 * child > 0: node of the tree, <= 0: leaf -child), node thresholds, nnodes + 1 leaves; feature f: 12 rect ints,
 * 3 weights, tilted flag. */
NV_API int nv_debug_cascade_tree(const nv_cascade *c, int tree, int cap_nodes, int *nnodes, int *feat_left_right,
                                 float *node_thr, float *leaves);
NV_API int nv_debug_cascade_feature(const nv_cascade *c, int feature, int rects12[12], float weights3[3], int *tilted);
/* LBP cascades: the 256-bit subset (eight words, bit `code` set: go to the first child) of internal node `node`, nodes
 * counted over all weak classifiers in file order; the cell rect of an LBP feature is rects12[0..3] above. */
NV_API int nv_debug_cascade_subset(const nv_cascade *c, int node, int subset8[8]);

NV_API int nv_debug_num_levels(nv_ctx *ctx);
NV_API int nv_debug_level_info(nv_ctx *ctx, int level, nv_level_info *info);
NV_API int nv_debug_get_gray(nv_ctx *ctx, uint8_t *dst, int cap_bytes, int *width, int *height);
NV_API int nv_debug_get_integral(nv_ctx *ctx, int level, int32_t *sum, uint32_t *sqsum);     /* (h+1)*(w+1) each */
NV_API int nv_debug_get_tilted(nv_ctx *ctx, int level, int32_t *tilted);                      /* (h+1)*(w+1); cascades with tilted features */
NV_API int nv_debug_get_depth_map(nv_ctx *ctx, int level, int16_t *depth);                    /* ny*nx           */
NV_API int nv_debug_get_candidates(nv_ctx *ctx, nv_rect *out, int cap, int *n);               /* raw, canonical order */
/* counters of the last call: [0] windows visited, [1] windows alive after stage 0,
 * [2] raw candidates, [3] kernels launched, [4..7] reserved */
NV_API int nv_debug_get_counters(nv_ctx *ctx, long long *out8);

#ifdef __cplusplus
}
#endif
#endif /* NUBOVCA_H */
