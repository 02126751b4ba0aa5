// K1: BGR -> gray -> 5x5 binomial blur -> uint8 plane + per-frame 256-bin histogram.
//
// Replaces cv2.cvtColor(BGR2GRAY) + cv2.GaussianBlur((5,5),0) (lane_detector.py:69,72) and the
// counting half of np.median (lane_detector.py:79).  Integer-exact (SURVEY.md A.1-A.3):
//   gray = (3735 B + 19235 G + 9798 R + 2^14) >> 15
//   blur = (sum_ij w_i w_j gray[y+i-2][x+j-2] + 128) >> 8,  w = [1 4 6 4 1], BORDER_REFLECT_101
#include <algorithm>

#include "lane_common.cuh"

namespace {

__device__ __forceinline__ int fold101(int p, int len)
{
    if (len == 1) return 0;
    while (p < 0 || p >= len) p = p < 0 ? -p : 2 * len - p - 2;
    return p;
}

__device__ __forceinline__ uint32_t gray_of(uint32_t b, uint32_t g, uint32_t r)
{
    return (3735u * b + 19235u * g + 9798u * r + (1u << 14)) >> 15;
}

constexpr int TW = 64, TH = 32, NT = 256;

// One CTA per 64 x 32 tile of a frame, any H, W.  Blurred frames of widths and heights the fused edge kernel
// (k1_fused.cu) does not take run here.
__global__ void __launch_bounds__(NT) k1_tile(const uint8_t *__restrict__ frames, uint8_t *__restrict__ blur,
                                              uint32_t *__restrict__ hist, int H, int W)
{
    __shared__ uint8_t g[TH + 4][TW + 4];
    __shared__ uint16_t hs[TH + 4][TW];
    __shared__ uint32_t lh[256];
    const int tid = threadIdx.x;
    const int f = blockIdx.z, x0 = blockIdx.x * TW, y0 = blockIdx.y * TH;
    const uint8_t *src = frames + (size_t)f * H * W * 3;
    lh[tid] = 0;
    for (int i = tid; i < (TH + 4) * (TW + 4); i += NT) {
        int ly = i / (TW + 4), lx = i - ly * (TW + 4);
        int gy = fold101(y0 + ly - 2, H), gx = fold101(x0 + lx - 2, W);
        const uint8_t *p = src + ((size_t)gy * W + gx) * 3;
        g[ly][lx] = (uint8_t)gray_of(p[0], p[1], p[2]);
    }
    __syncthreads();
    for (int i = tid; i < (TH + 4) * TW; i += NT) {
        int ly = i / TW, lx = i - ly * TW;
        const uint8_t *r = &g[ly][lx];
        hs[ly][lx] = (uint16_t)(r[0] + r[4] + 4 * (r[1] + r[3]) + 6 * r[2]);
    }
    __syncthreads();
    uint8_t *dst = blur + (size_t)f * H * W;
    for (int i = tid; i < TH * TW; i += NT) {
        int ly = i / TW, lx = i - ly * TW;
        int y = y0 + ly, x = x0 + lx;
        if (y < H && x < W) {
            uint32_t s = hs[ly][lx] + hs[ly + 4][lx] + 4u * (hs[ly + 1][lx] + hs[ly + 3][lx]) + 6u * hs[ly + 2][lx];
            uint32_t v = (s + 128u) >> 8;
            dst[(size_t)y * W + x] = (uint8_t)v;
            atomicAdd(&lh[v], 1u);
        }
    }
    __syncthreads();
    if (lh[tid]) atomicAdd(&hist[f * 256 + tid], lh[tid]);
}

// gray plane + histogram without the blur (scene_classifier.py:145-146 runs cv2.Canny on the plain grayscale frame)
__global__ void __launch_bounds__(256) k1_gray_hist(const uint8_t *__restrict__ frames, uint8_t *__restrict__ out,
                                                    uint32_t *__restrict__ hist, int P)
{
    __shared__ uint32_t lh[256];
    const int f = blockIdx.y, tid = threadIdx.x;
    lh[tid] = 0;
    __syncthreads();
    const uint8_t *src = frames + (size_t)f * P * 3;
    uint8_t *dst = out + (size_t)f * P;
    for (int i = blockIdx.x * 256 + tid; i < P; i += gridDim.x * 256) {
        const uint32_t v = gray_of(src[3 * i], src[3 * i + 1], src[3 * i + 2]);
        dst[i] = (uint8_t)v;
        atomicAdd(&lh[v], 1u);
    }
    __syncthreads();
    if (lh[tid]) atomicAdd(&hist[f * 256 + tid], lh[tid]);
}

__global__ void k_gray(const uint8_t *__restrict__ frame, uint8_t *__restrict__ gray, int n)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) gray[i] = (uint8_t)gray_of(frame[3 * i], frame[3 * i + 1], frame[3 * i + 2]);
}

}  // namespace

void launch_blur_hist(const uint8_t *frames, uint8_t *blur_out, uint32_t *hist, int n, int H, int W,
                      cudaStream_t st, int *launches, int blur)
{
    cudaMemsetAsync(hist, 0, sizeof(uint32_t) * 256 * n, st);
    if (!blur) {
        dim3 grid(std::min((H * W + 255) / 256, 1184), n);
        k1_gray_hist<<<grid, 256, 0, st>>>(frames, blur_out, hist, H * W);
    } else {
        dim3 grid((W + TW - 1) / TW, (H + TH - 1) / TH, n);
        k1_tile<<<grid, NT, 0, st>>>(frames, blur_out, hist, H, W);
    }
    *launches += 1;
}

void launch_gray_debug(const uint8_t *frame, uint8_t *gray, int H, int W, cudaStream_t st)
{
    int n = H * W;
    k_gray<<<(n + 255) / 256, 256, 0, st>>>(frame, gray, n);
}
