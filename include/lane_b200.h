/*
 * lane_b200.h -- C ABI of the B200-native batched lane-detection path.
 *
 * Drop-in boundary for ONE hot path of the reference:
 *   /root/reference/src/perception/lane_detector.py:178-218  LaneDetector.detect
 *   /root/reference/src/perception/lane_detector.py:253-272  LaneDetector.get_lane_center_offset
 * The reference has no FFI of its own (pure Python over cv2/numpy); the entry points below
 * are what a ctypes binding inside lane_detector.py binds (see INTEGRATION.md).  Each one
 * names the reference lines it replaces.
 *
 * Conventions: plain pointers and sizes only; every function returns 0 on success or a
 * negative lane_status code, never throws; the library never frees or reallocates caller
 * memory; one context per (device, stream); a context is not re-entrant.  All device work
 * of a call is enqueued on the context's stream; the blocking calls synchronise that
 * stream before returning.
 */
#ifndef LANE_B200_H
#define LANE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define LANE_API __attribute__((visibility("default")))
#else
#define LANE_API
#endif

#define LANE_B200_ABI_VERSION 1
#define LANE_NUM_POINTS 50          /* lane_detector.py:164  np.linspace(.., .., 50) */

typedef enum lane_status {
    LANE_OK = 0,
    LANE_ERR_INVALID = -1,          /* bad argument (shape, null pointer, batch too large, device index out of range) */
    LANE_ERR_CUDA = -2,             /* a CUDA runtime call or kernel failed; see lane_last_error */
    LANE_ERR_NO_DEVICE = -3,        /* no CUDA device visible, or (lane_ctx_create) not sm_100: there is NO CPU fallback */
    LANE_ERR_STATE = -4,            /* ROI / LUT not set before detect */
    LANE_ERR_UNSUPPORTED = -5       /* frame larger than this build supports */
} lane_status;

/* One side of one frame -- mirrors LaneLine (lane_detector.py:13-19). */
typedef struct lane_side {
    int32_t valid;                  /* 0 => the reference returns None for this side */
    int32_t n_lines;                /* segments that fed the fit (confidence = min(1, n/10)) */
    double raw[3];                  /* np.polyfit(y, x, 2) output, highest power first (:156) */
    double coeffs[3];               /* after the EMA with the previous fit (:159-161) -> LaneLine.polynomial */
    double confidence;              /* :171 */
    int32_t points[LANE_NUM_POINTS][2]; /* (x, y) int32, truncation toward zero (:164-167) -> LaneLine.points */
} lane_side;

/* Result record of one frame. */
typedef struct lane_record {
    lane_side side[2];              /* 0 = left, 1 = right (:206-216) */
    double offset;                  /* get_lane_center_offset (:253-272); meaningful iff offset_valid */
    int32_t offset_valid;
    int32_t median_x2;              /* 2 * np.median(blurred) (:79) */
    int32_t low, high;              /* Canny thresholds (:80-81) */
    int32_t n_edges;                /* non-zero pixels of the full-frame Canny map (:83) */
    int32_t n_roi_points;           /* non-zero pixels after the ROI mask (:89) */
    int32_t n_segments;             /* segments HoughLinesP returned (:94-101) */
    int32_t hysteresis_rounds;      /* propagation rounds the frame needed (diagnostic) */
    int32_t flags;                  /* LANE_FLAG_* */
    int32_t n_segments_found;       /* segments HoughLinesP found; > n_segments iff LANE_FLAG_SEGMENTS_TRUNCATED */
} lane_record;

#define LANE_FLAG_SEGMENTS_TRUNCATED 1   /* more segments than max_segments: extra ones dropped */
#define LANE_FLAG_POINTS_TRUNCATED 2     /* a side had more segments than its capacity (= max_segments) */

typedef struct lane_ctx lane_ctx;

/* ---- lifetime ------------------------------------------------------------------------ */
/* Replaces LaneDetector.__init__ (lane_detector.py:35-45) for a fixed frame size.
 * max_batch frames of height x width BGR can be processed per call.  max_segments bounds the
 * HoughLinesP output kept per frame (0 => default 256). */
LANE_API int lane_ctx_create(int device, int height, int width, int max_batch, int max_segments, lane_ctx **out);
LANE_API void lane_ctx_destroy(lane_ctx *ctx);
/* Message of the last failure on this context (or of the last failed create when ctx is NULL). */
LANE_API const char *lane_last_error(const lane_ctx *ctx);
LANE_API int lane_abi_version(void);

/* ---- static per-detector inputs ------------------------------------------------------- */
/* ROI mask produced once on the host by cv2.fillPoly (lane_detector.py:47-64): uint8[height*width],
 * non-zero = inside.  Replaces the per-frame _get_roi_mask/_apply_roi (:86-90).  May be called again on a live
 * context; if such a call fails, detect calls return LANE_ERR_STATE until one succeeds. */
LANE_API int lane_set_roi_mask(lane_ctx *ctx, const uint8_t *mask);
/* One ROI mask per camera of a rig (lane_detector.py:47-64, one LaneDetector(roi_vertices=...) per camera):
 * uint8[n_masks][height*width], non-zero = inside.  Mask r belongs to stream r: with n_masks > 1 frame f of a detect
 * call uses mask stream_id[f] (mask 0 when stream_id is NULL), and a call with n_streams > n_masks is refused with
 * LANE_ERR_INVALID.  A frame's records, taps and Hough outputs equal those of a context set with its mask alone.
 * n_masks = 1 is lane_set_roi_mask.  Re-setting and failures behave as for lane_set_roi_mask. */
LANE_API int lane_set_roi_masks(lane_ctx *ctx, const uint8_t *masks, int n_masks);
/* low/high Canny thresholds for every possible 2*median (index 0..510), filled by evaluating the
 * reference's own float64 expressions (lane_detector.py:80-81). */
LANE_API int lane_set_threshold_lut(lane_ctx *ctx, const uint8_t *low511, const uint8_t *high511);
/* HoughLinesP literals (lane_detector.py:94-101); defaults 50, 50, 150. */
LANE_API int lane_set_hough_params(lane_ctx *ctx, int threshold, int min_line_length, int max_line_gap);
/* smoothing_factor and (1 - smoothing_factor) exactly as the host evaluates them (:159-161). */
LANE_API int lane_set_smoothing(lane_ctx *ctx, double factor, double one_minus_factor);
/* gaussian_blur = 0 skips cv2.GaussianBlur (lane_detector.py:72): Canny then runs on the plain grayscale plane, as
 * the reference's SceneClassifier does (src/tagging/scene_classifier.py:145-146).  Default 1. */
LANE_API int lane_set_preprocess(lane_ctx *ctx, int gaussian_blur);
/* Keep per-stage intermediates of the next detect calls for the lane_debug_* taps (costs memory traffic). */
LANE_API int lane_set_debug(lane_ctx *ctx, int keep_intermediates);

/* ---- the hot path --------------------------------------------------------------------- */
/* Replaces n sequential LaneDetector.detect calls (lane_detector.py:178-218) plus
 * get_lane_center_offset (:253-272).
 *   frames            uint8 [n][height][width][3] BGR, C-contiguous; host memory when
 *                     frames_on_device == 0 (copied inside the call), device memory otherwise.
 *   stream_id         host int32[n], camera stream of each frame (NULL => all stream 0); frames of
 *                     one stream must appear in temporal order.
 *   n_streams         number of streams S.
 *   prev_fit          host double [S][2][3], in/out: prev_left_fit / prev_right_fit per stream (:43-44).
 *   prev_valid        host uint8 [S][2], in/out: 0 => None.
 *   out               host lane_record[n].
 * Blocking: returns after the records are in `out`. */
LANE_API int lane_detect_batch(lane_ctx *ctx, const uint8_t *frames, int frames_on_device, int n,
                      const int32_t *stream_id, int n_streams, double *prev_fit, uint8_t *prev_valid,
                      lane_record *out);

/* Same as lane_detect_batch for frames still in the decoder's NV12 layout (uint8 [n][height*3/2][width]): only
 * 1.5 B/px cross PCIe, the NV12 -> BGR conversion of lane_nv12_to_bgr_batch runs on the device chunk by chunk behind
 * the copies, and the records equal those of lane_detect_batch on the converted frames. */
LANE_API int lane_detect_batch_nv12(lane_ctx *ctx, const uint8_t *frames_nv12, int frames_on_device, int n,
                           const int32_t *stream_id, int n_streams, double *prev_fit, uint8_t *prev_valid,
                           lane_record *out);

/* Frame layouts a detect / ingest call accepts (what a decoder or VideoDataLoader hands out); lane_bgr_to_yuv420_batch
 * produces the two YUV ones (what an encoder takes). */
#define LANE_INPUT_BGR  0           /* uint8 [n][src_h][src_w][3] */
#define LANE_INPUT_NV12 1           /* uint8 [n][src_h*3/2][src_w], Y then interleaved UV (hardware decoders) */
#define LANE_INPUT_I420 2           /* uint8 [n][src_h*3/2][src_w], Y, then U plane, then V plane (software decoders) */

/* lane_detect_batch on frames of another size and/or layout, as VideoDataLoader.read_frame delivers them
 * (/root/reference/data/loaders/video_loader.py:96-131: decode, then cv2.resize(frame, target_size) at :108, :128) to
 * LaneDetector.detect (lane_detector.py:178-218).  Each frame becomes the context's height x width BGR frame on the device
 * -- cv2.resize(cv2.cvtColor(f, COLOR_YUV2BGR_NV12 | COLOR_YUV2BGR_I420), (width, height)) in one kernel for YUV, the
 * lane_resize_batch kernel for BGR -- and the usual path runs on it: only the source bytes cross PCIe, and the records
 * equal those of lane_detect_batch on the cv2-prepared frames.  format: LANE_INPUT_*; src_h / src_w: the frames' own
 * size (even for NV12 / I420).  Other arguments as for lane_detect_batch. */
LANE_API int lane_detect_batch_ingest(lane_ctx *ctx, const uint8_t *frames, int frames_on_device, int n, int format,
                                      int src_h, int src_w, const int32_t *stream_id, int n_streams, double *prev_fit,
                                      uint8_t *prev_valid, lane_record *out);

/* Asynchronous split of the above for pipelined callers: enqueue (device frames only; records
 * land in an internal pinned buffer), then collect (waits for the OLDEST batch in flight and returns
 * its records and the EMA state after it).
 *   prev_fit / prev_valid given:  the batch starts from that state; one batch in flight at a time.
 *   prev_fit = prev_valid = NULL: the batch continues from the state the previous batch left on the
 *       device (the streaming case: the detector object's prev_*_fit simply stays on the GPU), and a
 *       second batch may be queued behind the first -- enqueue, enqueue, collect, enqueue, collect, ...
 *       -- so the device never waits for the host between batches.  Batches run in order on one stream. */
LANE_API int lane_detect_enqueue(lane_ctx *ctx, const uint8_t *frames_dev, int n, const int32_t *stream_id,
                        int n_streams, const double *prev_fit, const uint8_t *prev_valid);
LANE_API int lane_detect_collect(lane_ctx *ctx, double *prev_fit, uint8_t *prev_valid, lane_record *out);

/* The context's CUDA stream (cudaStream_t as void*), so callers can record events on it. */
LANE_API void *lane_ctx_stream(lane_ctx *ctx);
/* Device copy of the records lane_detect_collect / lane_detect_batch returned last (lane_record[n]).  It stays valid
 * until the batch AFTER the next one is enqueued (two result slots alternate), so a multi-GPU caller can hand it to
 * NCCL without a host round trip (SURVEY.md 8e: the path's only collective is the gather of these records); the slot's next
 * writer must be ordered behind that read: lane_ctx_fence_records. */
LANE_API const lane_record *lane_ctx_records_device(lane_ctx *ctx);
/* Tell the context that work already enqueued on `reader_stream` (a cudaStream_t: the collective that gathers the records
 * of the batch collected last, SURVEY.md 8e) reads lane_ctx_records_device: only the kernel that next WRITES that result slot
 * (the fit of the batch after next) waits for it -- the edge kernels of the following batches do not.  Call it right after
 * enqueuing the reader. */
LANE_API int lane_ctx_fence_records(lane_ctx *ctx, void *reader_stream);
/* Use a caller-owned stream (cudaStream_t) instead of the context's own. */
LANE_API int lane_ctx_set_stream(lane_ctx *ctx, void *cuda_stream);

/* Which kernel family the last batch ran on (bit set = the fast path; a cleared bit means the launch was not possible
 * for this geometry or was rejected by the device, and the generic kernels produced the same results more slowly). */
#define LANE_PATH_FUSED_EDGE 1      /* one fused gray + blur + histogram + Sobel + NMS kernel (aligned widths) */
#define LANE_PATH_CLUSTER_CANNY 2   /* hysteresis + ROI + point list in one thread-block cluster per frame */
#define LANE_PATH_PPHT_DSMEM 4      /* HoughLinesP accumulator in distributed shared memory */
LANE_API int lane_ctx_last_paths(lane_ctx *ctx);

/* ---- measurement ---------------------------------------------------------------------- */
#define LANE_STAGE_H2D 0
#define LANE_STAGE_BLUR_HIST 1      /* K1: gray + 5x5 blur + histogram */
#define LANE_STAGE_CANNY 2          /* K2: thresholds + Sobel + NMS + hysteresis */
#define LANE_STAGE_COMPACT 3        /* ROI mask + ordered point list */
#define LANE_STAGE_PPHT 4           /* K4: HoughLinesP */
#define LANE_STAGE_FIT 5            /* K5: split + polyfit + EMA + points + offset */
#define LANE_STAGE_D2H 6
#define LANE_NUM_STAGES 7
/* When enabled, CUDA events bracket every stage of the next calls. */
LANE_API int lane_set_profiling(lane_ctx *ctx, int enabled);
/* Device time (ms) of each stage in the last completed call, and kernel launches it made. */
LANE_API int lane_get_stage_ms(lane_ctx *ctx, float ms[LANE_NUM_STAGES], int32_t launches[LANE_NUM_STAGES]);

/* ---- verification taps (need lane_set_debug(ctx, 1) before the detect call) ------------ */
#define LANE_TAP_BLUR 1             /* uint8 [H][W]   cv2.GaussianBlur output (:72) */
#define LANE_TAP_HIST 2             /* uint32[256]    histogram behind np.median (:79) */
#define LANE_TAP_CLASS 3            /* uint8 [H][W]   0 none / 1 weak / 2 strong before hysteresis */
#define LANE_TAP_EDGES 4            /* uint8 [H][W]   cv2.Canny output 0/255 (:83) */
#define LANE_TAP_POINTS 5           /* int32 [n_roi_points][2] (x,y) row-major order of masked edges (:89) */
#define LANE_TAP_SEGMENTS 6         /* int32 [n_segments][4] HoughLinesP output (:94-101) */
#define LANE_TAP_GRAY 7             /* uint8 [H][W]   cv2.cvtColor output (:69); recomputed on demand */
/* Copies tap `what` of frame `frame_index` of the last batch to host memory; *bytes_written is set. */
LANE_API int lane_debug_tap(lane_ctx *ctx, int what, int frame_index, void *host_out, size_t capacity,
                   size_t *bytes_written);

/* Standard Hough accumulator (BASELINE.json north-star add-on; what cv2.HoughLines(img,1,pi/180,t)
 * votes into) of the ROI-masked edge map of frame `frame_index` of the last batch:
 * int32 [182][2*(W+H)+3] with cv2's one-cell padding.  peaks (optional): int32 triples
 * (rho_index, angle_index, votes) of local maxima above `threshold` in cv2's output order. */
LANE_API int lane_hough_accumulator(lane_ctx *ctx, int frame_index, int32_t *accum_host, int threshold,
                           int32_t *peaks_host, int max_peaks, int *n_peaks);

/* The same for EVERY frame of the last batch in one call, without debug mode (north-star kernel #3: "Hough voting with
 * warp-aggregated shared-memory accumulators per theta band, followed by peak extraction"): votes come from the ROI rows
 * of the frames' Canny bit-planes, peaks are extracted and ordered on the device.
 *   peaks_host    int32 [n][max_peaks][3]  (rho_index, angle_index, votes) per frame in cv2.HoughLines order
 *                 (votes descending, ties by ascending accumulator index); only the first min(n_peaks, max_peaks) rows
 *                 of a frame are written (if more were found, which ones are kept is unspecified)
 *   n_peaks_host  int32 [n]                peaks found per frame
 *   accum_host    optional int32 [n][182][2*(W+H)+3]  the padded accumulators (verification: 4.4 MB per 1080p frame)
 *   device_ms     optional: device time of the voting + peak kernels for the whole batch */
LANE_API int lane_hough_lines_batch(lane_ctx *ctx, int threshold, int max_peaks, int32_t *peaks_host,
                           int32_t *n_peaks_host, int32_t *accum_host, float *device_ms);

/* Edge pixels of the Canny map inside the rectangle [x0,x1) x [y0,y1), for every frame of the last batch (int32[n]):
 * SceneClassifier's centre-region edge density, np.sum(edges[h//3:2*h//3, w//3:2*w//3] > 0)
 * (/root/reference/src/tagging/scene_classifier.py:148-150), as a popcount on the device. */
LANE_API int lane_edge_count_rect(lane_ctx *ctx, int x0, int y0, int x1, int y1, int32_t *counts_host);

/* ---- frame ingest (SURVEY.md 8f rank 1: the step before the path) -------------------------------------------
 * Replaces the pixel work of VideoDataLoader.read_frame / read_frame_at
 * (/root/reference/data/loaders/video_loader.py:96-131): `frame = cv2.resize(frame, self.target_size)` (:108, :128),
 * OpenCV's default INTER_LINEAR on uint8, for a whole batch of equally sized frames, bit-exact.
 * src: uint8 [n][src_h][src_w][channels], dst: uint8 [n][dst_h][dst_w][channels], channels = 1 or 3, both dense.
 * on_device = 1: both are device pointers on `device`, the kernel is enqueued on `cuda_stream` (a cudaStream_t,
 * NULL = default stream) and the call returns without synchronising -- this is how resized frames are handed to
 * lane_detect_batch(frames_on_device = 1) without ever leaving HBM.  on_device = 0: both are host pointers, the
 * call copies in, resizes, copies out and synchronises.  Needs no context; errors via lane_last_error(NULL). */
LANE_API int lane_resize_batch(const uint8_t *src, int n, int src_h, int src_w, int channels, uint8_t *dst, int dst_h,
                               int dst_w, int on_device, int device, void *cuda_stream);

/* NV12 -> BGR for a batch of decoded frames, bit-exact against cv2.cvtColor(nv12, cv2.COLOR_YUV2BGR_NV12): what a
 * hardware decoder hands out (Y plane + interleaved half-resolution UV plane, 1.5 B/px) becomes the BGR frame
 * VideoDataLoader.read_frame returns (/root/reference/data/loaders/video_loader.py:103-110).
 * src: uint8 [n][height*3/2][width], dst: uint8 [n][height][width][3]; width and height even.  on_device / device /
 * cuda_stream as for lane_resize_batch.  Needs no context; errors via lane_last_error(NULL). */
LANE_API int lane_nv12_to_bgr_batch(const uint8_t *src, int n, int height, int width, uint8_t *dst, int on_device,
                                    int device, void *cuda_stream);

/* Decoder output at camera resolution -> the frame VideoDataLoader.read_frame returns with target_size set
 * (/root/reference/data/loaders/video_loader.py:96-131): per frame
 * cv2.resize(cv2.cvtColor(f, COLOR_YUV2BGR_NV12 | COLOR_YUV2BGR_I420), (dst_w, dst_h)), bit-exact, in one pass that
 * reads the 1.5 B/px source and writes only the destination (the full-resolution BGR frame is never stored).
 * src: uint8 [n][src_h*3/2][src_w] in `format` (LANE_INPUT_NV12 or LANE_INPUT_I420), src_h / src_w even;
 * dst: uint8 [n][dst_h][dst_w][3], any positive size (equal to the source size: conversion only).  on_device / device /
 * cuda_stream as for lane_resize_batch.  Needs no context; errors via lane_last_error(NULL). */
LANE_API int lane_yuv420_to_bgr_batch(const uint8_t *src, int format, int n, int src_h, int src_w, uint8_t *dst,
                                      int dst_h, int dst_w, int on_device, int device, void *cuda_stream);

/* ---- frame egress (SURVEY.md 8f rank 3: the step after the overlays when annotated video is written) ---------------
 * cv2.cvtColor(f, COLOR_BGR2YUV_I420) per frame (NV12: the same samples, U and V interleaved), for annotated frames
 * that are in device memory -- what LaneDetector.draw_lanes (lane_detector.py:220-251) and the offset indicator leave in
 * HBM, ready for an encoder (libx264 -pix_fmt yuv420p, a hardware encoder's NV12 surface) at 1.5 B/px.
 * src_dev: device uint8 [n][height][width][3]; dst: uint8 [n][height*3/2][width],
 * device memory (dst_on_device = 1: enqueued on cuda_stream, returns without synchronising) or host memory
 * (dst_on_device = 0: converted chunk by chunk, each chunk copied out while the next is converted; blocking).
 * format: LANE_INPUT_I420 or LANE_INPUT_NV12; height, width even; n = 0 does nothing.  Host sources are not taken
 * (cv2.cvtColor converts those where they are).  Needs no context; errors via lane_last_error(NULL). */
LANE_API int lane_bgr_to_yuv420_batch(const uint8_t *src_dev, int format, int n, int height, int width, uint8_t *dst,
                                      int dst_on_device, int device, void *cuda_stream);

/* ---- scene statistics (SURVEY.md 8f rank 2, second half) -----------------------------------------------------
 * Integer sums behind SceneClassifier's image cues (/root/reference/src/tagging/scene_classifier.py):
 *   avg_brightness = np.mean(cvtColor(frame, BGR2GRAY))                       (:237-238)  = sum_gray / (H*W)
 *   laplacian_var  = cv2.Laplacian(gray, cv2.CV_64F).var()                    (:254)      = E[L^2] - E[L]^2
 *   green_ratio    = sum(inRange(cvtColor(frame, BGR2HSV), (35,40,40), (85,255,255)) > 0) / size   (:183-186)
 * The device returns exact integers; the caller forms the float64 quantities (see scene_stats.py). */
typedef struct lane_frame_stat {
    uint64_t sum_gray;              /* sum of the BGR2GRAY plane */
    int64_t sum_laplacian;          /* sum of L = 3x3 Laplacian (ksize 1, BORDER_REFLECT_101) of the gray plane */
    uint64_t sum_laplacian_sq;      /* sum of L*L */
    uint64_t green_pixels;          /* pixels with 35 <= H <= 85, S >= 40, V >= 40 in OpenCV's 8-bit HSV */
} lane_frame_stat;
/* frames: uint8 [n][height][width][3] BGR, host (on_device = 0) or device pointer; out: n records in host memory.
 * Blocking (synchronises `cuda_stream`).  Needs no context; errors via lane_last_error(NULL). */
LANE_API int lane_frame_stats(const uint8_t *frames, int on_device, int n, int height, int width, lane_frame_stat *out,
                              int device, void *cuda_stream);

/* ---- drawing (SURVEY.md 8f ranks 3 and 4: the step after the path, and its input fixture) -----------------------------
 * Batched, bit-exact device forms of the OpenCV drawing calls the reference makes on every frame:
 *   LaneDetector.draw_lanes                      /root/reference/src/perception/lane_detector.py:220-251
 *   OverlayRenderer.draw_lane_offset_indicator   /root/reference/src/visualization/overlays.py:103-148
 *   SyntheticDataGenerator.generate_*            /root/reference/data/generators/__pycache__/synthetic_data.cpython-312.pyc
 * frames: uint8 [n][height][width][3] BGR, drawn IN PLACE; device pointer when on_device = 1 (work enqueued on
 * `cuda_stream`), host pointer otherwise (copied in, drawn, copied back).  Both calls return after the stream has been
 * synchronised.  device_ms (optional): device time of the command upload + rasterisation.  Need no context; errors via
 * lane_last_error(NULL). */

/* A stream of cv2-level drawing calls per frame, executed in order (painter's order, as consecutive cv2 calls are).
 * commands: int32 words; command_begin: int64 [n + 1], frame f owns words [command_begin[f], command_begin[f + 1]).
 * color = b | g << 8 | r << 16.  Every command reproduces OpenCV 4.13 for uint8 images, LINE_8, shift 0:
 *   LANE_DRAW_LINE              x1 y1 x2 y2 color thickness                cv2.line
 *   LANE_DRAW_RECTANGLE         x1 y1 x2 y2 color thickness(<0: filled)    cv2.rectangle
 *   LANE_DRAW_CIRCLE            cx cy radius color thickness(<0 only)      cv2.circle, filled
 *   LANE_DRAW_FILLPOLY          color npts x0 y0 x1 y1 ...                 cv2.fillPoly(img, [pts], color)
 *   LANE_DRAW_POLYLINES         color thickness closed npts x0 y0 ...      cv2.polylines(img, [pts], closed, color, thickness)
 *   LANE_DRAW_FILLPOLY_WEIGHTED color alpha beta gamma(float32 bits) npts x0 y0 ...
 *                               o = img.copy(); cv2.fillPoly(o, [pts], color); img = cv2.addWeighted(img, alpha, o, beta, gamma)
 *                               (gamma must be 0, as everywhere in the reference: cv2's scalar tail rounds otherwise)
 *   LANE_DRAW_BITMAP            x y w h color bits[h][(w + 31) / 32]       pixels (x + i, y + j) with bit i of row j set get
 *                               `color` (how cv2.putText output enters: rendered once per string on the host)
 *   LANE_DRAW_ROWS              y_start count x1 x2 color[count]           cv2.line((x1, y), (x2, y), color[y - y_start], 1)
 *                               for count consecutive rows (the generator's sky gradient) */
#define LANE_DRAW_LINE 1
#define LANE_DRAW_RECTANGLE 2
#define LANE_DRAW_CIRCLE 3
#define LANE_DRAW_FILLPOLY 4
#define LANE_DRAW_POLYLINES 5
#define LANE_DRAW_FILLPOLY_WEIGHTED 6
#define LANE_DRAW_BITMAP 7
#define LANE_DRAW_ROWS 8
LANE_API int lane_draw_commands(uint8_t *frames, int on_device, int n, int height, int width, const int32_t *commands,
                                const int64_t *command_begin, int device, void *cuda_stream, float *device_ms);

/* SyntheticDataGenerator.generate_frame_with_vehicles (the reference's data/generators/__pycache__/synthetic_data.cpython-312.pyc,
 * SURVEY.md Appendix B) for frame_count = frame_count0 .. frame_count0 + n - 1: the scene (sky gradient, ground, road triangle,
 * lane dashes, trees, 2-4 vehicles drawn from NumPy's legacy RandomState(frame_count % 100)) is laid out by the library's host
 * code and rasterised by the same kernel; frames are overwritten (zeroed first), bit-identical to the Python / cv2 generator. */
LANE_API int lane_generate_frames(uint8_t *frames, int on_device, int n, int height, int width, int64_t frame_count0,
                                  int device, void *cuda_stream, float *device_ms);

/* LaneDetector.draw_lanes (lane_detector.py:220-251) for a batch: the lane area between the two 50-point polylines
 * filled with (0, 255, 100) at weight 0.3 (only when fill_lane and both sides are valid), then the left polyline in
 * (255, 0, 0) and the right one in (0, 0, 255), thickness 3.
 *   left_points / right_points   host int32 [n][LANE_NUM_POINTS][2] (x, y) = LaneLine.points (lane_side.points)
 *   left_valid / right_valid     host uint8 [n], 0 = that side is None */
LANE_API int lane_draw_lanes_batch(uint8_t *frames, int on_device, int n, int height, int width, const int32_t *left_points,
                                   const uint8_t *left_valid, const int32_t *right_points, const uint8_t *right_valid,
                                   int fill_lane, int device, void *cuda_stream, float *device_ms);
/* The same straight from the lane records on the device (lane_ctx_records_device of the batch collected last, or any
 * device copy of lane_record[n]): no lane data touches the host.  frames_dev: device pointer, drawn in place; the kernel is
 * enqueued on `cuda_stream` and the call returns without synchronising. */
LANE_API int lane_draw_lanes_records(uint8_t *frames_dev, int n, int height, int width, const lane_record *records_dev,
                                     int fill_lane, int device, void *cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* LANE_B200_H */
