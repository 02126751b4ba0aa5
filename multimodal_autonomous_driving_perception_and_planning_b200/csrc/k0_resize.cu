// K0: batched bilinear resize of uint8 frames, bit-exact with cv2.resize(frame, target_size) (INTER_LINEAR).
//
// SURVEY.md 8(f) rank 1 -- the step before the lane path: VideoDataLoader.read_frame / read_frame_at
// (/root/reference/data/loaders/video_loader.py:96-131) resize every decoded frame with cv2.resize (:108, :128).
// Arithmetic per oracle/resize.py (OpenCV's 8-bit bilinear: 11-bit fixed-point taps from float32 fractions,
// horizontal pass in int, vertical pass ((b*(H>>4))>>16 summed, +2, >>2)).  The tap tables depend only on the two
// geometries; the host computes them once with the same float32 operations OpenCV uses and caches them per device.
//
// Bound: HBM (reads the touched source pixels once, writes the destination once; no arithmetic to speak of).
#include <math.h>

#include <map>
#include <mutex>
#include <string>
#include <tuple>
#include <vector>

#include "host_stage.h"
#include "k0_common.cuh"

namespace {

std::mutex g_mu;
std::map<std::tuple<int, int, int, int, int>, ResizeTaps> g_taps;

void frac(int d, double scale, int *s, float *f)
{
    float fx = (float)((d + 0.5) * scale - 0.5);
    int sx = (int)floorf(fx);
    *s = sx;
    *f = fx - (float)sx;
}

short coef(float v) { return (short)lrintf(v * 2048.f); }      // cvRound (nearest even) of a float32 product

cudaError_t build_taps(int sh, int sw, int dh, int dw, ResizeTaps *t)
{
    std::vector<int> xo(dw);
    std::vector<short2> al(dw), be(dh);
    std::vector<int2> yo(dh);
    const double scale_x = 1.0 / ((double)dw / sw), scale_y = 1.0 / ((double)dh / sh);
    for (int d = 0; d < dw; d++) {
        int s; float f;
        frac(d, scale_x, &s, &f);
        if (s < 0) { f = 0; s = 0; }
        if (s >= sw - 1) { f = 0; s = sw - 1; }
        xo[d] = s;
        al[d] = make_short2(coef(1.f - f), coef(f));
    }
    for (int d = 0; d < dh; d++) {
        int s; float f;
        frac(d, scale_y, &s, &f);
        yo[d] = make_int2(std::min(std::max(s, 0), sh - 1), std::min(std::max(s + 1, 0), sh - 1));
        be[d] = make_short2(coef(1.f - f), coef(f));
    }
    cudaError_t e;
    if ((e = cudaMalloc(&t->xofs, sizeof(int) * dw))) return e;
    if ((e = cudaMalloc(&t->alpha, sizeof(short2) * dw))) return e;
    if ((e = cudaMalloc(&t->yofs, sizeof(int2) * dh))) return e;
    if ((e = cudaMalloc(&t->beta, sizeof(short2) * dh))) return e;
    if ((e = cudaMemcpy(t->xofs, xo.data(), sizeof(int) * dw, cudaMemcpyHostToDevice))) return e;
    if ((e = cudaMemcpy(t->alpha, al.data(), sizeof(short2) * dw, cudaMemcpyHostToDevice))) return e;
    if ((e = cudaMemcpy(t->yofs, yo.data(), sizeof(int2) * dh, cudaMemcpyHostToDevice))) return e;
    return cudaMemcpy(t->beta, be.data(), sizeof(short2) * dh, cudaMemcpyHostToDevice);
}

// One thread = PX consecutive destination pixels of one row (PX * CN bytes, written with the widest stores the
// alignment allows); a warp covers a contiguous run of the row, so the source reads of a warp fall in two short
// row segments that stay in L1 across the PX pixels.
template <int CN, int PX>
__global__ void __launch_bounds__(256) k0_resize(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst,
                                                 const int *__restrict__ xofs, const short2 *__restrict__ alpha,
                                                 const int2 *__restrict__ yofs, const short2 *__restrict__ beta,
                                                 int sh, int sw, int dh, int dw)
{
    const int dx0 = (blockIdx.x * blockDim.x + threadIdx.x) * PX, dy = blockIdx.y, f = blockIdx.z;
    if (dx0 >= dw) return;
    const int2 yy = __ldg(yofs + dy);
    const short2 b = __ldg(beta + dy);
    const uint8_t *r0 = src + ((size_t)f * sh + yy.x) * sw * CN, *r1 = src + ((size_t)f * sh + yy.y) * sw * CN;
    uint8_t *out = dst + (((size_t)f * dh + dy) * dw + dx0) * CN;
    uint8_t px[PX * CN];
#pragma unroll
    for (int k = 0; k < PX; k++) {
        const int dx = min(dx0 + k, dw - 1);
        const int x0 = __ldg(xofs + dx), x1 = min(x0 + 1, sw - 1);
        const short2 a = __ldg(alpha + dx);
#pragma unroll
        for (int c = 0; c < CN; c++) {
            const int h0 = (int)__ldg(r0 + x0 * CN + c) * a.x + (int)__ldg(r0 + x1 * CN + c) * a.y;
            const int h1 = (int)__ldg(r1 + x0 * CN + c) * a.x + (int)__ldg(r1 + x1 * CN + c) * a.y;
            px[k * CN + c] = (uint8_t)k0_vmix(h0, h1, b.x, b.y);
        }
    }
    if (dx0 + PX <= dw && ((uintptr_t)out & 3) == 0 && (PX * CN) % 4 == 0) {
#pragma unroll
        for (int q = 0; q < PX * CN / 4; q++)
            reinterpret_cast<uint32_t *>(out)[q] = (uint32_t)px[4 * q] | ((uint32_t)px[4 * q + 1] << 8) |
                                                   ((uint32_t)px[4 * q + 2] << 16) | ((uint32_t)px[4 * q + 3] << 24);
    } else {
        for (int k = 0; k < PX && dx0 + k < dw; k++)
            for (int c = 0; c < CN; c++) out[k * CN + c] = px[k * CN + c];
    }
}

}  // namespace

cudaError_t lane_resize_taps(int sh, int sw, int dh, int dw, ResizeTaps *t)
{
    int device = 0;
    cudaError_t e;
    if ((e = cudaGetDevice(&device))) return e;
    std::lock_guard<std::mutex> lk(g_mu);
    const auto key = std::make_tuple(device, sh, sw, dh, dw);
    auto it = g_taps.find(key);
    if (it != g_taps.end()) {
        *t = it->second;
        return cudaSuccess;
    }
    if ((e = build_taps(sh, sw, dh, dw, t))) return e;
    g_taps[key] = *t;
    return cudaSuccess;
}

void launch_resize(const uint8_t *src, uint8_t *dst, int n, int channels, int sh, int sw, int dh, int dw,
                   const ResizeTaps &t, cudaStream_t st)
{
    constexpr int PX = 4;
    dim3 grid((dw + 256 * PX - 1) / (256 * PX), dh, n);
    if (channels == 3)
        k0_resize<3, PX><<<grid, 256, 0, st>>>(src, dst, t.xofs, t.alpha, t.yofs, t.beta, sh, sw, dh, dw);
    else
        k0_resize<1, PX><<<grid, 256, 0, st>>>(src, dst, t.xofs, t.alpha, t.yofs, t.beta, sh, sw, dh, dw);
}

extern "C" int lane_resize_batch(const uint8_t *src, int n, int src_h, int src_w, int channels, uint8_t *dst, int dst_h,
                                 int dst_w, int on_device, int device, void *cuda_stream)
{
    constexpr const char *who = "lane_resize_batch";
    if (!src || !dst || n <= 0 || src_h <= 0 || src_w <= 0 || dst_h <= 0 || dst_w <= 0 || (channels != 1 && channels != 3))
        return lane_api_fail(LANE_ERR_INVALID, who, "bad arguments (uint8 frames with 1 or 3 channels, positive sizes)");
    if (dst_h > 65535 || n > 65535) return lane_api_fail(LANE_ERR_UNSUPPORTED, who, "destination height / batch above 65535");
    if (int rc = lane_api_device(who, device)) return rc;
    cudaError_t e;
    ResizeTaps t;
    if ((e = lane_resize_taps(src_h, src_w, dst_h, dst_w, &t))) return lane_api_fail(LANE_ERR_CUDA, who, "tap tables", e);
    cudaStream_t st = (cudaStream_t)cuda_stream;
    auto launch = [&](const uint8_t *s, uint8_t *d) {
        launch_resize(s, d, n, channels, src_h, src_w, dst_h, dst_w, t, st);
        const cudaError_t r = cudaGetLastError();
        return r ? lane_api_fail(LANE_ERR_CUDA, who, "kernel launch", r) : LANE_OK;
    };
    if (on_device) return launch(src, dst);
    return lane_host_round_trip(who, device, st, src, (size_t)n * src_h * src_w * channels, dst,
                                (size_t)n * dst_h * dst_w * channels, launch);
}
