// K0c: decoder output at camera resolution -> the frame the lane path runs on, in one pass (SURVEY.md 8f rank 1).
//
// VideoDataLoader.read_frame / read_frame_at (/root/reference/data/loaders/video_loader.py:96-131) decode a frame and
// cv2.resize it to target_size (:108, :128) before LaneDetector.detect sees it.  For YUV 4:2:0 decoder output this
// kernel produces, per destination pixel, exactly
//     cv2.resize(cv2.cvtColor(src, COLOR_YUV2BGR_NV12 | COLOR_YUV2BGR_I420), (dw, dh))      (INTER_LINEAR)
// The conversion is per pixel, so the resize may convert its two source rows x two source columns on the fly (from Y
// and the 2x2 block's (U, V), k0_common.cuh) and apply k0_resize's 11-bit horizontal taps and vertical step to them:
// the full-resolution BGR frame is never written.  HBM-bound: reads the touched 1.5 B/px of the source once, writes
// 3 B per destination pixel.
//
// K0e: raw camera frames (8-bit Bayer mosaics, 1 B/px) the same way: per destination pixel
//     cv2.resize(cv2.cvtColor(src, COLOR_Bayer{RGGB,BGGR,GRBG,GBRG}2BGR), (dw, dh))      (INTER_LINEAR)
// with the two source rows x two source columns of every tap demosaiced from their 4x4 raw neighbourhood
// (k0_bayer_resize_px).  A frame at the destination size runs on identity taps: the demosaic alone.
//
// K0f: packed YUV 4:2:2 camera frames (UYVY / YUYV, 2 B/px) the same way as K0c: per destination pixel
//     cv2.resize(cv2.cvtColor(src, COLOR_YUV2BGR_UYVY | COLOR_YUV2BGR_YUY2), (dw, dh))      (INTER_LINEAR)
// with the two source rows x two source columns of every tap converted from their Y and their pair's (U, V)
// (k0_yuv422_resize_px).  At the destination size launch_ingest takes k0_nv12.cu's conversion kernels instead.
#include "host_stage.h"
#include "k0_common.cuh"

namespace {

using namespace k0yuv;

// k0_resize's thread shape: one thread = PX consecutive destination pixels of one row, packed 4-byte stores when
// aligned, byte stores otherwise; a warp covers a contiguous run of the row, so its source reads (two short source row
// segments, and for 4:2:0 the chroma rows under them) stay in L1 across the PX pixels.  FMT: the layout
// (LANE_INPUT_NV12 / I420 / UYVY / YUYV, or LANE_INPUT_BAYER_RGGB for every Bayer pattern, read at run-time `phase`:
// lane_bayer_phase).
template <int FMT, int PX>
__global__ void __launch_bounds__(256) k0_ingest_resize(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst,
                                                        const int *__restrict__ xofs, const short2 *__restrict__ alpha,
                                                        const int2 *__restrict__ yofs, const short2 *__restrict__ beta,
                                                        int sh, int sw, int dh, int dw, int phase)
{
    const int dx0 = (blockIdx.x * blockDim.x + threadIdx.x) * PX, dy = blockIdx.y, f = blockIdx.z;
    if (dx0 >= dw) return;
    const int2 yy = __ldg(yofs + dy);
    const short2 b = __ldg(beta + dy);
    const uint8_t *s = src + lane_input_frame_bytes(FMT, sh, sw, f);
    uint8_t *out = dst + (((size_t)f * dh + dy) * dw + dx0) * 3;
    uint8_t o[PX * 3];
    if constexpr (lane_input_bayer(FMT))
        k0_bayer_resize_px<PX>(s, sh, sw, phase, yy, b, xofs, alpha, dx0, dw, o);
    else if constexpr (lane_input_yuv422(FMT))
        k0_yuv422_resize_px<PX>(s, sw, lane_yuv422_y0(FMT), yy, b, xofs, alpha, dx0, dw, o);
    else
        k0_yuv420_resize_px<FMT, PX>(s, sh, sw, yy, b, xofs, alpha, dx0, dw, o);
    k0_store_px<3, PX>(out, o, dx0, dw);
}

// The frames of a rig: every frame has its own descriptor (layout, size, tap tables), so cameras of different
// resolutions and decoders share one launch.  The grid is k0_ingest_resize's; a block reads its frame's descriptor
// once, and the branch on the layout is uniform over the block.  A frame already at dh x dw runs on identity taps,
// which reproduce the source (BGR) or cv2.cvtColor's frame (YUV, Bayer) exactly.
//
// The Bayer, the packed 4:2:2 and the BGR / YUV 4:2:0 pixel work are separate functions kept out of line: inlined side
// by side the first and the last need 60 registers, which would drop the kernel from 5 to 4 blocks per SM; apart, each
// fits the kernel's 48.
template <int PX>
__device__ __noinline__ void rig_bgr_yuv420(const RigFrame &d, int2 yy, short2 b, int dx0, int dw, uint8_t *out)
{
    uint8_t o[PX * 3];
    if (d.format == LANE_INPUT_BGR) {
        const uint8_t *r0 = d.src + (size_t)yy.x * d.sw * 3, *r1 = d.src + (size_t)yy.y * d.sw * 3;
        k0_resize_px<3, PX>(r0, r1, d.xofs, d.alpha, b, d.sw, dx0, dw, o);
    } else if (d.format == LANE_INPUT_NV12) {
        k0_yuv420_resize_px<LANE_INPUT_NV12, PX>(d.src, d.sh, d.sw, yy, b, d.xofs, d.alpha, dx0, dw, o);
    } else {
        k0_yuv420_resize_px<LANE_INPUT_I420, PX>(d.src, d.sh, d.sw, yy, b, d.xofs, d.alpha, dx0, dw, o);
    }
    k0_store_px<3, PX>(out, o, dx0, dw);
}

template <int PX>
__device__ __noinline__ void rig_bayer(const RigFrame &d, int2 yy, short2 b, int dx0, int dw, uint8_t *out)
{
    uint8_t o[PX * 3];
    k0_bayer_resize_px<PX>(d.src, d.sh, d.sw, lane_bayer_phase(d.format), yy, b, d.xofs, d.alpha, dx0, dw, o);
    k0_store_px<3, PX>(out, o, dx0, dw);
}

// The frame's layout picks a constant Y0 offset: with the offset a run-time value in the addresses the branch needs 64
// registers.
template <int PX>
__device__ __noinline__ void rig_yuv422(const RigFrame &d, int2 yy, short2 b, int dx0, int dw, uint8_t *out)
{
    uint8_t o[PX * 3];
    if (lane_yuv422_y0(d.format))
        k0_yuv422_resize_px<PX>(d.src, d.sw, 1, yy, b, d.xofs, d.alpha, dx0, dw, o);
    else
        k0_yuv422_resize_px<PX>(d.src, d.sw, 0, yy, b, d.xofs, d.alpha, dx0, dw, o);
    k0_store_px<3, PX>(out, o, dx0, dw);
}

template <int PX>
__global__ void __launch_bounds__(256) k0_rig_ingest(const RigFrame *__restrict__ frames, uint8_t *__restrict__ dst, int dh,
                                                     int dw)
{
    __shared__ RigFrame d;
    const int dx0 = (blockIdx.x * blockDim.x + threadIdx.x) * PX, dy = blockIdx.y, f = blockIdx.z;
    if (threadIdx.x == 0) d = frames[f];
    __syncthreads();
    if (dx0 >= dw) return;
    const int2 yy = __ldg(d.yofs + dy);
    const short2 b = __ldg(d.beta + dy);
    uint8_t *out = dst + (((size_t)f * dh + dy) * dw + dx0) * 3;
    if (lane_input_bayer(d.format))
        rig_bayer<PX>(d, yy, b, dx0, dw, out);
    else if (lane_input_yuv422(d.format))
        rig_yuv422<PX>(d, yy, b, dx0, dw, out);
    else
        rig_bgr_yuv420<PX>(d, yy, b, dx0, dw, out);
}

}  // namespace

cudaError_t rig_frame(const uint8_t *src, int format, int sh, int sw, int dh, int dw, RigFrame *d)
{
    ResizeTaps t;
    const cudaError_t e = lane_resize_taps(sh, sw, dh, dw, &t);
    if (e) return e;
    *d = RigFrame{src, format, sh, sw, t.xofs, t.alpha, t.yofs, t.beta};
    return cudaSuccess;
}

void launch_rig_ingest(const RigFrame *frames_dev, int n, uint8_t *dst, int dh, int dw, cudaStream_t st)
{
    constexpr int PX = 4;
    const dim3 grid((dw + 256 * PX - 1) / (256 * PX), dh, n);
    k0_rig_ingest<PX><<<grid, 256, 0, st>>>(frames_dev, dst, dh, dw);
}

cudaError_t launch_ingest(const uint8_t *src, int format, int n, int sh, int sw, uint8_t *dst, int dh, int dw,
                          cudaStream_t st)
{
    if (!lane_input_resizes(format, sh, sw, dh, dw)) {            // INTER_LINEAR at scale 1 is the identity
        if (lane_input_yuv422(format))
            launch_yuv422_to_bgr(src, format, dst, n, sh, sw, st);
        else
            launch_yuv420_to_bgr(src, format, dst, n, sh, sw, st);
        return cudaGetLastError();
    }
    ResizeTaps t;
    cudaError_t e = lane_resize_taps(sh, sw, dh, dw, &t);
    if (e) return e;
    if (format == LANE_INPUT_BGR) {
        launch_resize(src, dst, n, 3, sh, sw, dh, dw, t, st);
        return cudaGetLastError();
    }
    constexpr int PX = 4;
    const dim3 grid((dw + 256 * PX - 1) / (256 * PX), dh, n);
    auto launch = [&](auto kernel) {
        kernel<<<grid, 256, 0, st>>>(src, dst, t.xofs, t.alpha, t.yofs, t.beta, sh, sw, dh, dw, lane_bayer_phase(format));
    };
    switch (format) {
    case LANE_INPUT_NV12: launch(k0_ingest_resize<LANE_INPUT_NV12, PX>); break;
    case LANE_INPUT_I420: launch(k0_ingest_resize<LANE_INPUT_I420, PX>); break;
    case LANE_INPUT_UYVY: launch(k0_ingest_resize<LANE_INPUT_UYVY, PX>); break;
    case LANE_INPUT_YUYV: launch(k0_ingest_resize<LANE_INPUT_YUYV, PX>); break;
    default: launch(k0_ingest_resize<LANE_INPUT_BAYER_RGGB, PX>);
    }
    return cudaGetLastError();
}

namespace {

// The context-free conversion entries: n frames of a layout `accepts` takes (`formats` names them), checked against
// the layout table, become BGR at dst_h x dst_w on the device or through a host round trip.  `who` starts every message.
int to_bgr(const char *who, bool (*accepts)(int), const char *formats, const uint8_t *src, int format, int n, int src_h,
           int src_w, uint8_t *dst, int dst_h, int dst_w, int on_device, int device, void *cuda_stream)
{
    if (!src || !dst || n < 1 || src_h < 1 || src_w < 1 || dst_h < 1 || dst_w < 1)
        return lane_api_fail(LANE_ERR_INVALID, who, "bad arguments (non-null pointers, positive sizes)");
    if (!accepts(format)) return lane_api_fail(LANE_ERR_INVALID, who, formats);
    if (const char *why = lane_input_refusal(format, src_h, src_w)) return lane_api_fail(LANE_ERR_INVALID, who, why);
    if (lane_input_resizes(format, src_h, src_w, dst_h, dst_w) && (dst_h > 65535 || n > 65535))
        return lane_api_fail(LANE_ERR_UNSUPPORTED, who, "destination height / batch above 65535");
    if (int rc = lane_api_device(who, device)) return rc;
    cudaStream_t st = (cudaStream_t)cuda_stream;
    auto launch = [&](const uint8_t *s, uint8_t *d) {
        const cudaError_t e = launch_ingest(s, format, n, src_h, src_w, d, dst_h, dst_w, st);
        return e ? lane_api_fail(LANE_ERR_CUDA, who, "launch", e) : LANE_OK;
    };
    if (on_device) return launch(src, dst);
    return lane_host_round_trip(who, device, st, src, lane_input_frame_bytes(format, src_h, src_w, n), dst,
                                (size_t)n * dst_h * dst_w * 3, launch);
}

}  // namespace

extern "C" int lane_yuv420_to_bgr_batch(const uint8_t *src, int format, int n, int src_h, int src_w, uint8_t *dst,
                                        int dst_h, int dst_w, int on_device, int device, void *cuda_stream)
{
    return to_bgr("lane_yuv420_to_bgr_batch", lane_input_yuv420, "format must be LANE_INPUT_NV12 or LANE_INPUT_I420", src,
                  format, n, src_h, src_w, dst, dst_h, dst_w, on_device, device, cuda_stream);
}

extern "C" int lane_bayer_to_bgr_batch(const uint8_t *src, int format, int n, int src_h, int src_w, uint8_t *dst,
                                       int dst_h, int dst_w, int on_device, int device, void *cuda_stream)
{
    return to_bgr("lane_bayer_to_bgr_batch", lane_input_bayer, "format must be a LANE_INPUT_BAYER_* layout", src, format,
                  n, src_h, src_w, dst, dst_h, dst_w, on_device, device, cuda_stream);
}

extern "C" int lane_yuv422_to_bgr_batch(const uint8_t *src, int format, int n, int src_h, int src_w, uint8_t *dst,
                                        int dst_h, int dst_w, int on_device, int device, void *cuda_stream)
{
    return to_bgr("lane_yuv422_to_bgr_batch", lane_input_yuv422, "format must be LANE_INPUT_UYVY or LANE_INPUT_YUYV", src,
                  format, n, src_h, src_w, dst, dst_h, dst_w, on_device, device, cuda_stream);
}

extern "C" int lane_nv12_to_bgr_batch(const uint8_t *src, int n, int height, int width, uint8_t *dst, int on_device,
                                      int device, void *cuda_stream)
{
    return to_bgr("lane_nv12_to_bgr_batch", lane_input_yuv420, "format must be LANE_INPUT_NV12 or LANE_INPUT_I420", src,
                  LANE_INPUT_NV12, n, height, width, dst, height, width, on_device, device, cuda_stream);
}
