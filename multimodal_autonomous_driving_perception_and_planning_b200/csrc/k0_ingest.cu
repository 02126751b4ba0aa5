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
#include "host_stage.h"
#include "k0_common.cuh"

namespace {

using namespace k0yuv;

// k0_resize's thread shape: one thread = PX consecutive destination pixels of one row, packed 4-byte stores when
// aligned, byte stores otherwise; a warp covers a contiguous run of the row, so its source reads (two short luma row
// segments and the chroma rows under them) stay in L1 across the PX pixels.
template <int FMT, int PX>
__global__ void __launch_bounds__(256) k0_yuv420_resize(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst,
                                                        const int *__restrict__ xofs, const short2 *__restrict__ alpha,
                                                        const int2 *__restrict__ yofs, const short2 *__restrict__ beta,
                                                        int sh, int sw, int dh, int dw)
{
    const int dx0 = (blockIdx.x * blockDim.x + threadIdx.x) * PX, dy = blockIdx.y, f = blockIdx.z;
    if (dx0 >= dw) return;
    const int2 yy = __ldg(yofs + dy);
    const short2 b = __ldg(beta + dy);
    const uint8_t *s = src + (size_t)f * sh * sw * 3 / 2;
    const uint8_t *l0 = s + (size_t)yy.x * sw, *l1 = s + (size_t)yy.y * sw;
    uint8_t *out = dst + (((size_t)f * dh + dy) * dw + dx0) * 3;
    uint8_t o[PX * 3];
#pragma unroll
    for (int k = 0; k < PX; k++) {
        const int dx = min(dx0 + k, dw - 1);
        const int x0 = __ldg(xofs + dx), x1 = min(x0 + 1, sw - 1);
        const short2 a = __ldg(alpha + dx);
        uint32_t p00[3], p01[3], p10[3], p11[3];     // BGR of (row y0 | y1) x (column x0 | x1)
        px(__ldg(l0 + x0), chroma<FMT>(s, sh, sw, yy.x >> 1, x0 >> 1), p00[0], p00[1], p00[2]);
        px(__ldg(l0 + x1), chroma<FMT>(s, sh, sw, yy.x >> 1, x1 >> 1), p01[0], p01[1], p01[2]);
        px(__ldg(l1 + x0), chroma<FMT>(s, sh, sw, yy.y >> 1, x0 >> 1), p10[0], p10[1], p10[2]);
        px(__ldg(l1 + x1), chroma<FMT>(s, sh, sw, yy.y >> 1, x1 >> 1), p11[0], p11[1], p11[2]);
#pragma unroll
        for (int c = 0; c < 3; c++) {
            const int h0 = (int)p00[c] * a.x + (int)p01[c] * a.y;
            const int h1 = (int)p10[c] * a.x + (int)p11[c] * a.y;
            o[k * 3 + c] = (uint8_t)k0_vmix(h0, h1, b.x, b.y);
        }
    }
    if (dx0 + PX <= dw && ((uintptr_t)out & 3) == 0 && (PX * 3) % 4 == 0) {
#pragma unroll
        for (int q = 0; q < PX * 3 / 4; q++)
            reinterpret_cast<uint32_t *>(out)[q] = (uint32_t)o[4 * q] | ((uint32_t)o[4 * q + 1] << 8) |
                                                   ((uint32_t)o[4 * q + 2] << 16) | ((uint32_t)o[4 * q + 3] << 24);
    } else {
        for (int k = 0; k < PX && dx0 + k < dw; k++)
            for (int c = 0; c < 3; c++) out[k * 3 + c] = o[k * 3 + c];
    }
}

}  // namespace

cudaError_t launch_ingest(const uint8_t *src, int format, int n, int sh, int sw, uint8_t *dst, int dh, int dw,
                          cudaStream_t st)
{
    if (format != LANE_INPUT_BGR && sh == dh && sw == dw) {       // INTER_LINEAR at scale 1 is the identity
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
    if (format == LANE_INPUT_I420)
        k0_yuv420_resize<LANE_INPUT_I420, PX><<<grid, 256, 0, st>>>(src, dst, t.xofs, t.alpha, t.yofs, t.beta, sh, sw, dh, dw);
    else
        k0_yuv420_resize<LANE_INPUT_NV12, PX><<<grid, 256, 0, st>>>(src, dst, t.xofs, t.alpha, t.yofs, t.beta, sh, sw, dh, dw);
    return cudaGetLastError();
}

namespace {

int yuv420_to_bgr(const char *who, const uint8_t *src, int format, int n, int src_h, int src_w, uint8_t *dst, int dst_h,
                  int dst_w, int on_device, int device, void *cuda_stream)
{
    if (!src || !dst || n < 1 || src_h < 1 || src_w < 1 || dst_h < 1 || dst_w < 1)
        return lane_api_fail(LANE_ERR_INVALID, who, "bad arguments (non-null pointers, positive sizes)");
    if (format != LANE_INPUT_NV12 && format != LANE_INPUT_I420)
        return lane_api_fail(LANE_ERR_INVALID, who, "format must be LANE_INPUT_NV12 or LANE_INPUT_I420");
    if ((src_h | src_w) & 1) return lane_api_fail(LANE_ERR_INVALID, who, "YUV 4:2:0 needs even width and height");
    const bool resize = dst_h != src_h || dst_w != src_w;
    if (resize && (dst_h > 65535 || n > 65535))
        return lane_api_fail(LANE_ERR_UNSUPPORTED, who, "destination height / batch above 65535");
    if (int rc = lane_api_device(who, device)) return rc;
    cudaStream_t st = (cudaStream_t)cuda_stream;
    auto launch = [&](const uint8_t *s, uint8_t *d) {
        const cudaError_t e = launch_ingest(s, format, n, src_h, src_w, d, dst_h, dst_w, st);
        return e ? lane_api_fail(LANE_ERR_CUDA, who, "launch", e) : LANE_OK;
    };
    if (on_device) return launch(src, dst);
    return lane_host_round_trip(who, device, st, src, (size_t)n * src_h * src_w * 3 / 2, dst, (size_t)n * dst_h * dst_w * 3,
                                launch);
}

}  // namespace

extern "C" int lane_yuv420_to_bgr_batch(const uint8_t *src, int format, int n, int src_h, int src_w, uint8_t *dst,
                                        int dst_h, int dst_w, int on_device, int device, void *cuda_stream)
{
    return yuv420_to_bgr("lane_yuv420_to_bgr_batch", src, format, n, src_h, src_w, dst, dst_h, dst_w, on_device, device,
                         cuda_stream);
}

extern "C" int lane_nv12_to_bgr_batch(const uint8_t *src, int n, int height, int width, uint8_t *dst, int on_device,
                                      int device, void *cuda_stream)
{
    return yuv420_to_bgr("lane_nv12_to_bgr_batch", src, LANE_INPUT_NV12, n, height, width, dst, height, width, on_device,
                         device, cuda_stream);
}
