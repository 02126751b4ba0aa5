// Shared pieces of the frame-ingest kernels (K0): the YUV 4:2:0 -> BGR arithmetic of k0_nv12.cu / k0_ingest.cu, its
// inverse for the egress kernel (k8_egress.cu) and the INTER_LINEAR tap tables and vertical step of k0_resize.cu.
#pragma once
#include "lane_common.cuh"

// ---- YUV 4:2:0 -> BGR, bit-exact with cv2.cvtColor(f, COLOR_YUV2BGR_NV12 / COLOR_YUV2BGR_I420) ----------------------
// ITU-R BT.601 limited range, 20-bit fixed point, arithmetic shift, saturation (oracle/nv12.py restates it).  NV12 and
// I420 carry the same samples and differ only in where U and V are stored.
namespace k0yuv {

constexpr int CY = 1220542, CUB = 2116026, CUG = -409993, CVG = -852492, CVR = 1673527, SHIFT = 20;

__device__ __forceinline__ uint32_t sat8(int v) { return (uint32_t)min(max(v, 0), 255); }

struct UV {
    int r, g, b;                       // chroma terms of one 2x2 block (rounding constant included)
};

__device__ __forceinline__ UV uv_terms(int u, int v)
{
    u -= 128; v -= 128;
    UV t;
    t.r = (1 << (SHIFT - 1)) + CVR * v;
    t.g = (1 << (SHIFT - 1)) + CVG * v + CUG * u;
    t.b = (1 << (SHIFT - 1)) + CUB * u;
    return t;
}

__device__ __forceinline__ void px(int yv, const UV &t, uint32_t &b, uint32_t &g, uint32_t &r)
{
    const int y = max(0, yv - 16) * CY;
    b = sat8((y + t.b) >> SHIFT); g = sat8((y + t.g) >> SHIFT); r = sat8((y + t.r) >> SHIFT);
}

// Chroma terms of block (by, bx) of frame `s` (H x W luma, both even).
//   NV12: interleaved (U, V) pairs at H*W + by*W + 2*bx
//   I420: U plane at H*W, V plane at H*W*5/4, each with pitch W/2
template <int FMT>
__device__ __forceinline__ UV chroma(const uint8_t *s, int H, int W, int by, int bx)
{
    const size_t P = (size_t)H * W;
    if constexpr (FMT == LANE_INPUT_NV12) {
        const uint8_t *p = s + P + (size_t)by * W + 2 * bx;
        return uv_terms(__ldg(p), __ldg(p + 1));
    } else {
        const size_t q = P + (size_t)by * (W / 2) + bx;
        return uv_terms(__ldg(s + q), __ldg(s + q + P / 4));
    }
}

// ---- BGR -> YUV 4:2:0, bit-exact with cv2.cvtColor(f, COLOR_BGR2YUV_I420) (k8_egress.cu) ---------------------------
// The same BT.601 limited range in 20-bit fixed point with a round-half constant; Y from every pixel, U and V from the
// top-left pixel of each 2x2 block (no averaging).  All sums are non-negative, so >> is a floor.
constexpr int EYR = 269484, EYG = 528482, EYB = 102760;
constexpr int EUR = -155188, EUG = -305135, EUB = 460324;
constexpr int EVR = 460324, EVG = -385875, EVB = -74448;
constexpr int EY0 = (16 << SHIFT) + (1 << (SHIFT - 1)), EC0 = (128 << SHIFT) + (1 << (SHIFT - 1));

__device__ __forceinline__ uint32_t bgr_y(int b, int g, int r) { return sat8((EYR * r + EYG * g + EYB * b + EY0) >> SHIFT); }
__device__ __forceinline__ uint32_t bgr_u(int b, int g, int r) { return sat8((EUR * r + EUG * g + EUB * b + EC0) >> SHIFT); }
__device__ __forceinline__ uint32_t bgr_v(int b, int g, int r) { return sat8((EVR * r + EVG * g + EVB * b + EC0) >> SHIFT); }

}  // namespace k0yuv

// ---- cv2.resize INTER_LINEAR on uint8 (oracle/resize.py) -------------------------------------------------------------
// Tap tables of one (source, destination) geometry, device memory.  Built once per (device, geometry) with the float32
// operations OpenCV uses and cached for the life of the process.
struct ResizeTaps {
    int *xofs = nullptr;        // [dw]   first source column
    short2 *alpha = nullptr;    // [dw]   (a0, a1); the second tap is min(x0 + 1, sw - 1)
    int2 *yofs = nullptr;       // [dh]   the two source rows, clamped one by one
    short2 *beta = nullptr;     // [dh]   (b0, b1) from the unclamped fraction
};

// vertical step: ((b*(H>>4))>>16 summed, +2, >>2), saturated
__device__ __forceinline__ uint32_t k0_vmix(int h0, int h1, int b0, int b1)
{
    const int v = (((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2;
    return (uint32_t)min(v, 255);
}

// Tables for the current device (cached; the first call of a geometry allocates and uploads them synchronously).
cudaError_t lane_resize_taps(int sh, int sw, int dh, int dw, ResizeTaps *t);
// k0_resize over n dense frames of `channels` (1 or 3) uint8 planes; device pointers, enqueued on st, no checks.
void launch_resize(const uint8_t *src, uint8_t *dst, int n, int channels, int sh, int sw, int dh, int dw,
                   const ResizeTaps &t, cudaStream_t st);

// k0_nv12: YUV 4:2:0 -> BGR at the source size
void launch_yuv420_to_bgr(const uint8_t *src, int format, uint8_t *dst, int n, int H, int W, cudaStream_t st);

// ---- ingest: any LANE_INPUT_* layout at any size -> BGR at dh x dw --------------------------------------------------
// NV12 / I420 at the destination size: k0_nv12's conversion kernels; NV12 / I420 at another size: the fused
// conversion + resize kernel (k0_ingest.cu); BGR at another size: k0_resize.  BGR at its own size needs no kernel and is
// not taken.  Device pointers, enqueued on st; the caller has validated the sizes (even YUV sizes, grid limits).
cudaError_t launch_ingest(const uint8_t *src, int format, int n, int sh, int sw, uint8_t *dst, int dh, int dw,
                          cudaStream_t st);
