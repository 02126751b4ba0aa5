// K6: per-frame image statistics of the reference's SceneClassifier, exact integer sums (SURVEY.md 8f rank 2).
//
//   _analyze_conditions (/root/reference/src/tagging/scene_classifier.py:237-257):
//       gray = cv2.cvtColor(frame, BGR2GRAY); avg_brightness = np.mean(gray)                     (:237-238)
//       laplacian_var = cv2.Laplacian(gray, cv2.CV_64F).var()                                    (:254)
//   _classify_road_type (:183-186):
//       hsv = cv2.cvtColor(frame, BGR2HSV); green = cv2.inRange(hsv, (35,40,40), (85,255,255))
//       green_ratio = np.sum(green > 0) / green.size
//
// The device returns integers only -- sum(gray), sum(L), sum(L^2) of the 3x3 Laplacian L (kernel [0 1 0; 1 -4 1;
// 0 1 0], BORDER_REFLECT_101) and the count of green pixels -- so the host forms mean / variance / ratio in float64
// from exact numbers.  OpenCV's 8-bit HSV is integer arithmetic with two 12-bit fixed-point division tables
// (oracle/scene_stats.py restates it and is pinned against cv2); a pixel can only be green when G is the unique
// maximum over R (cv2 tests V == R first), so the hue is only evaluated there.
//
// Bound: HBM (3 B/px read, nothing written).  A CTA takes a 64x128 tile: gray of the tile and its one-pixel frame
// goes to shared memory once (gray sum and green test on the way), the Laplacian reads it back.
#include <math.h>
#include <stdlib.h>

#include <algorithm>
#include <type_traits>

#include <vector>

#include "host_stage.h"
#include "lane_common.cuh"

namespace {

constexpr int TR = 64, TC = 128, K6T = 256;

__device__ __forceinline__ int fold1(int p, int n)      // BORDER_REFLECT_101 for a one-pixel border
{
    if (n == 1) return 0;
    if (p < 0) return -p;
    if (p >= n) return 2 * n - 2 - p;
    return p;
}

__global__ void __launch_bounds__(K6T) k6_frame_stats(const uint8_t *__restrict__ frames, unsigned long long *__restrict__ acc,
                                                      int H, int W, const int *__restrict__ sdiv, const int *__restrict__ hdiv,
                                                      int h_lo, int h_hi, int s_lo, int v_lo)
{
    __shared__ uint8_t g[(TR + 2) * (TC + 2)];
    __shared__ unsigned long long red[4][K6T / 32];
    const int f = blockIdx.z, r0 = blockIdx.y * TR, c0 = blockIdx.x * TC, tid = threadIdx.x;
    const uint8_t *fr = frames + (size_t)f * H * W * 3;
    unsigned sum_g = 0, green = 0;
    for (int i = tid; i < (TR + 2) * (TC + 2); i += K6T) {
        const int lr = i / (TC + 2), lc = i - lr * (TC + 2);
        const int y = r0 + lr - 1, x = c0 + lc - 1;
        const bool inside = lr >= 1 && lr <= TR && lc >= 1 && lc <= TC && y < H && x < W;
        uint8_t gv = 0;
        if (y <= H && x <= W) {                                   // the frame of the last partial tile is still needed
            const uint8_t *p = fr + ((size_t)fold1(y, H) * W + fold1(x, W)) * 3;
            const int b = __ldg(p), gg = __ldg(p + 1), r = __ldg(p + 2);
            gv = (uint8_t)((3735 * b + 19235 * gg + 9798 * r + 16384) >> 15);       // cv2 BGR2GRAY, Q15
            if (inside) {
                sum_g += gv;
                if (gg > r && gg >= b && gg >= v_lo) {            // V == G and V != R: the only branch that can be green
                    const int diff = gg - min(b, r);
                    const int s = (diff * __ldg(sdiv + gg) + (1 << 11)) >> 12;
                    const int h = ((b - r + 2 * diff) * __ldg(hdiv + diff) + (1 << 11)) >> 12;   // >= 0 here
                    green += (s >= s_lo && h >= h_lo && h <= h_hi) ? 1u : 0u;
                }
            }
        }
        g[i] = gv;
    }
    __syncthreads();
    long long s1 = 0;
    unsigned long long s2 = 0;
    for (int i = tid; i < TR * TC; i += K6T) {
        const int lr = i / TC, lc = i - lr * TC;
        if (r0 + lr < H && c0 + lc < W) {
            const uint8_t *c = g + (lr + 1) * (TC + 2) + lc + 1;
            const int L = (int)c[-(TC + 2)] + (int)c[TC + 2] + (int)c[-1] + (int)c[1] - 4 * (int)c[0];
            s1 += L;
            s2 += (unsigned)(L * L);
        }
    }
    // block reduction of the four sums (s1 is carried as two's complement in the unsigned adder)
    unsigned long long v[4] = {sum_g, (unsigned long long)s1, s2, green};
#pragma unroll
    for (int k = 0; k < 4; k++)
        for (int o = 16; o; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
    if ((tid & 31) == 0)
        for (int k = 0; k < 4; k++) red[k][tid >> 5] = v[k];
    __syncthreads();
    if (tid < 4) {
        unsigned long long t = 0;
        for (int w = 0; w < K6T / 32; w++) t += red[tid][w];
        atomicAdd(&acc[(size_t)f * 4 + tid], t);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Strip form (W % 16 == 0, 16-byte aligned frames): the same sums with K1F's data path.  A warp owns a 512-px column
// strip (16 px per lane, three 16-byte loads per lane per row, lanes 0 / 31 are the one-pixel halo) and rolls down a
// band of rows in registers.  gray = 2 IDP2A per pixel as packed u16x2 pairs; the Laplacian is formed on the pairs as
// L' = up + down + left + right + 1020 - 4*centre (0..2040, carry-free), two rows of state alternating between two
// register slots; sum(gray) and sum(L') are IDP2A reductions, sum(L'^2) two IMADs per pair.  The green test needs
// G > R, G >= B, G >= 40: three signed byte dot products per pixel (IDP4A with +1/-1 selectors) whose sign bits are
// ORed; the rare survivors re-read their three bytes (L1 hits) and evaluate OpenCV's hue / saturation exactly.
constexpr int K6_SPX = 16, K6_STRIP = 30 * K6_SPX, K6_WARPS = 4;

__device__ __forceinline__ uint32_t k6_dp2a_lo(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t d;
    asm("dp2a.lo.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ uint32_t k6_dp2a_hi(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t d;
    asm("dp2a.hi.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ int k6_dp4a_us(uint32_t a, uint32_t b, int c)     // unsigned bytes of a times signed bytes of b
{
    int d;
    asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ uint4 k6_ldg(const uint4 *p)
{
    uint4 r;
    asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ void k6_gray16(const uint32_t (&w)[12], uint32_t (&g)[8])
{
    constexpr uint32_t CB = 2 * 3735, CG = 2 * 19235, CR = 2 * 9798, RND = 1u << 15;
    constexpr uint32_t KBG = CB | (CG << 16), KR0 = CR, K0B = CB << 16, KGR = CG | (CR << 16);
#pragma unroll
    for (int q = 0; q < 4; q++) {
        const uint32_t w0 = w[3 * q], w1 = w[3 * q + 1], w2 = w[3 * q + 2];
        const uint32_t s0 = k6_dp2a_hi(KR0, w0, k6_dp2a_lo(KBG, w0, RND));
        const uint32_t s1 = k6_dp2a_lo(KGR, w1, k6_dp2a_hi(K0B, w0, RND));
        const uint32_t s2 = k6_dp2a_lo(KR0, w2, k6_dp2a_hi(KBG, w1, RND));
        const uint32_t s3 = k6_dp2a_hi(KGR, w2, k6_dp2a_lo(K0B, w2, RND));
        g[2 * q] = __byte_perm(s0, s1, 0x7632);
        g[2 * q + 1] = __byte_perm(s2, s3, 0x7632);
    }
}

// sign bit set <=> pixel cannot be green: (G - R - 1) | (G - B), four pixels per three words (the V >= 40 test is left to
// the exact path: dark greenish pixels are rare and it saves a dot product per pixel here)
__device__ __forceinline__ uint32_t k6_not_green4(uint32_t w0, uint32_t w1, uint32_t w2)
{
    // bytes: w0 = B0 G0 R0 B1 | w1 = G1 R1 B2 G2 | w2 = R2 B3 G3 R3 ; selector bytes are signed (+1 = 0x01, -1 = 0xFF)
    const int a0 = k6_dp4a_us(w0, 0x00FF0100u, -1) | k6_dp4a_us(w0, 0x000001FFu, 0);
    const int a1 = k6_dp4a_us(w1, 0x0000FF01u, -1) | k6_dp4a_us(w1, 0x00000001u, k6_dp4a_us(w0, 0xFF000000u, 0));
    const int a2 = k6_dp4a_us(w2, 0x000000FFu, k6_dp4a_us(w1, 0x01000000u, -1)) | k6_dp4a_us(w1, 0x01FF0000u, 0);
    const int a3 = k6_dp4a_us(w2, 0xFF010000u, -1) | k6_dp4a_us(w2, 0x0001FF00u, 0);
    return ((uint32_t)a0 >> 31) | (((uint32_t)a1 >> 31) << 1) | (((uint32_t)a2 >> 31) << 2) | (((uint32_t)a3 >> 31) << 3);
}

__global__ void __launch_bounds__(K6_WARPS * 32, 5) k6_strip(const uint8_t *__restrict__ frames, unsigned long long *__restrict__ acc,
                                                             int *__restrict__ task_counter, int n_frames, int H, int W,
                                                             int band_rows, const int *__restrict__ sdiv,
                                                             const int *__restrict__ hdiv, int h_lo, int h_hi, int s_lo, int v_lo)
{
    const int lane = threadIdx.x & 31;
    const int n_strips = (W + K6_STRIP - 1) / K6_STRIP, n_bands = (H + band_rows - 1) / band_rows;
    const int n_tasks = n_frames * n_bands * n_strips;
    const size_t frame_px = (size_t)H * W;
    for (;;) {
        int task = 0;
        if (lane == 0) task = atomicAdd(task_counter, 1);
        task = __shfl_sync(0xffffffffu, task, 0);
        if (task >= n_tasks) break;
        const int strip = task % n_strips, band = (task / n_strips) % n_bands, f = task / (n_strips * n_bands);
        const int r0 = band * band_rows, r1 = min(r0 + band_rows, H);
        const int xl = strip * K6_STRIP - K6_SPX + K6_SPX * lane;
        const bool in_img = xl >= 0 && xl < W;
        const bool is_out = in_img && lane >= 1 && lane <= 30;
        const bool left_edge = xl == 0, right_edge = xl + K6_SPX == W;
        const uint8_t *src = frames + f * frame_px * 3 + (size_t)max(xl, 0) * 3;
        uint32_t gs[2][8], hs[2][8];                 // gray rows y-2 / y-1 and the horizontal part of row y-1, two slots
#pragma unroll
        for (int j = 0; j < 8; j++) gs[0][j] = gs[1][j] = hs[0][j] = hs[1][j] = 0;
        uint32_t sum_g = 0, sum_l = 0, green = 0;
        unsigned long long sum_l2 = 0;
        uint32_t w[12];
#pragma unroll
        for (int j = 0; j < 12; j++) w[j] = 0;
        auto load_row = [&](int y) {
            const int ya = abs(y), yy = min(ya, 2 * H - 2 - ya);       // BORDER_REFLECT_101, one-row halo, H >= 2
            if (in_img) {
                const uint4 *p = reinterpret_cast<const uint4 *>(src + (uint32_t)(yy * W) * 3u);
                const uint4 a = k6_ldg(p), b = k6_ldg(p + 1), c = k6_ldg(p + 2);
                w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
                w[8] = c.x; w[9] = c.y; w[10] = c.z; w[11] = c.w;
            }
        };
        load_row(r0 - 1);
        auto row_step = [&](auto slot, int y) {
            constexpr int k = decltype(slot)::value, o = k ^ 1;
            uint32_t g[8];
            k6_gray16(w, g);
            uint32_t ng = 0xFFFFu;                                   // "cannot be green" bits of this lane's 16 pixels
            const bool body_row = y >= r0 && y < r1;
            if (body_row && is_out) {
                ng = k6_not_green4(w[0], w[1], w[2]) | (k6_not_green4(w[3], w[4], w[5]) << 4) |
                     (k6_not_green4(w[6], w[7], w[8]) << 8) | (k6_not_green4(w[9], w[10], w[11]) << 12);
            }
            const int yra = abs(y), yrow = min(yra, 2 * H - 2 - yra);
            if (y + 1 <= r1) load_row(y + 1);
            // horizontal part of this row: left + right + 1020 - 4 * centre
            uint32_t L7 = __shfl_up_sync(0xffffffffu, g[7], 1), R0 = __shfl_down_sync(0xffffffffu, g[0], 1);
            if (left_edge) L7 = g[0];                                // x = -1 := x = 1 (high half of the first pair)
            if (right_edge) R0 = g[7];                               // x = W := x = W - 2 (low half of the last pair)
            uint32_t O[9];
            O[0] = __byte_perm(L7, g[0], 0x5432);
#pragma unroll
            for (int j = 1; j < 8; j++) O[j] = __byte_perm(g[j - 1], g[j], 0x5432);
            O[8] = __byte_perm(g[7], R0, 0x5432);
#pragma unroll
            for (int j = 0; j < 8; j++) hs[k][j] = O[j] + O[j + 1] + 0x03FC03FCu - 4u * g[j];
            if (is_out) {
                if (body_row) {
#pragma unroll
                    for (int j = 0; j < 8; j++) sum_g = k6_dp2a_lo(g[j], 0x0101u, sum_g);
                }
                if (y > r0 && y <= r1) {                              // Laplacian of row y-1: up = gs[k] (row y-2), down = g
                    uint32_t row_l2 = 0;
#pragma unroll
                    for (int j = 0; j < 8; j++) {
                        const uint32_t lp = hs[o][j] + gs[k][j] + g[j];
                        sum_l = k6_dp2a_lo(lp, 0x0101u, sum_l);
                        const uint32_t lo = lp & 0xFFFFu, hi = lp >> 16;
                        row_l2 += lo * lo + hi * hi;
                    }
                    sum_l2 += row_l2;
                }
            }
#pragma unroll
            for (int j = 0; j < 8; j++) gs[k][j] = g[j];             // slot k now holds row y (a rename, not a move)
            uint32_t cand = ~ng & 0xFFFFu;
            while (cand) {                                           // rare: exact hue / saturation of the survivors
                const int p = __ffs(cand) - 1;
                cand &= cand - 1;
                const uint8_t *q = src + ((size_t)yrow * W + p) * 3;
                const int b = __ldg(q), gg = __ldg(q + 1), r = __ldg(q + 2);
                const int diff = gg - min(b, r);
                const int s = (diff * __ldg(sdiv + gg) + (1 << 11)) >> 12;
                const int h = ((b - r + 2 * diff) * __ldg(hdiv + diff) + (1 << 11)) >> 12;
                green += (gg >= v_lo && s >= s_lo && h >= h_lo && h <= h_hi) ? 1u : 0u;
            }
        };
        for (int y = r0 - 1;;) {
            row_step(std::integral_constant<int, 0>{}, y);
            if (++y > r1) break;
            row_step(std::integral_constant<int, 1>{}, y);
            if (++y > r1) break;
        }
        // sum(L) = sum(L') - 1020 * px and sum(L^2) = sum(L'^2) - 2040 * sum(L') + 1020^2 * px are formed on the host
        unsigned long long v[4] = {sum_g, sum_l, sum_l2, green};
#pragma unroll
        for (int q = 0; q < 4; q++)
            for (int o2 = 16; o2; o2 >>= 1) v[q] += __shfl_xor_sync(0xffffffffu, v[q], o2);
        if (lane < 4) {
            const unsigned long long t = lane == 0 ? v[0] : lane == 1 ? v[1] : lane == 2 ? v[2] : v[3];
            if (t) atomicAdd(&acc[(size_t)f * 4 + lane], t);
        }
    }
}

}  // namespace

extern "C" int lane_frame_stats(const uint8_t *frames, int on_device, int n, int height, int width, lane_frame_stat *out,
                                int device, void *cuda_stream)
{
    constexpr const char *who = "lane_frame_stats";
    if (!frames || !out || n <= 0 || height <= 0 || width <= 0) return lane_api_fail(LANE_ERR_INVALID, who, "bad arguments");
    if (n > 65535) return lane_api_fail(LANE_ERR_UNSUPPORTED, who, "batch above 65535");
    if (int rc = lane_api_device(who, device)) return rc;
    cudaStream_t st = (cudaStream_t)cuda_stream;
    // OpenCV's tables: sdiv[i] = round(255*4096 / i), hdiv180[i] = round(180*4096 / (6*i)), entry 0 unused
    int h_tab[512] = {0};
    for (int i = 1; i < 256; i++) {
        h_tab[i] = (int)lrint((255 << 12) / (1. * i));
        h_tab[256 + i] = (int)lrint((180 << 12) / (6. * i));
    }
    std::vector<unsigned long long> h_acc((size_t)n * 4);
    bool strip = false;
    // device scratch: the tables, then the sums and the strip kernel's task counter
    const size_t scratch_bytes = 512 * sizeof(int) + ((size_t)n * 4 + 2) * sizeof(unsigned long long);
    auto launch = [&](const uint8_t *staged, uint8_t *scratch) {
        int *d_tab = reinterpret_cast<int *>(scratch);
        unsigned long long *d_acc = reinterpret_cast<unsigned long long *>(scratch + 512 * sizeof(int));
        const uint8_t *d_frames = on_device ? frames : staged;
        cudaError_t e = cudaMemcpyAsync(d_tab, h_tab, sizeof h_tab, cudaMemcpyHostToDevice, st);
        if (!e) e = cudaMemsetAsync(d_acc, 0, (size_t)n * 4 * sizeof(unsigned long long), st);
        if (e) return lane_api_fail(LANE_ERR_CUDA, who, "upload", e);
        dim3 grid((width + TC - 1) / TC, (height + TR - 1) / TR, n);
        if (grid.y > 65535) return lane_api_fail(LANE_ERR_UNSUPPORTED, who, "frame too tall");
        strip = width % 16 == 0 && ((uintptr_t)d_frames % 16) == 0 && height >= 2 &&
                (size_t)height * width * 3 < ((size_t)1 << 32);
        if (strip) {
            int sms = 0;
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
            int *d_counter = reinterpret_cast<int *>(d_acc + (size_t)n * 4);       // task counter, right behind the sums
            e = cudaMemsetAsync(d_counter, 0, sizeof(int), st);
            const int n_strips = (width + K6_STRIP - 1) / K6_STRIP, warps = sms * 5 * K6_WARPS;
            const long rows_per_warp = ((long)n * height * n_strips + 2 * warps - 1) / (2 * warps);
            const int band_rows = (int)std::max(12L, std::min(102L, rows_per_warp));
            k6_strip<<<sms * 5, K6_WARPS * 32, 0, st>>>(d_frames, d_acc, d_counter, n, height, width, band_rows, d_tab, d_tab + 256,
                                                        35, 85, 40, 40);
        } else {
            k6_frame_stats<<<grid, K6T, 0, st>>>(d_frames, d_acc, height, width, d_tab, d_tab + 256, 35, 85, 40, 40);
        }
        e = cudaGetLastError();
        if (!e) e = cudaMemcpyAsync(h_acc.data(), d_acc, h_acc.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st);
        return e ? lane_api_fail(LANE_ERR_CUDA, who, "kernel / download", e) : LANE_OK;
    };
    // host frames go in ahead of the scratch; the few sums come back in launch
    const int rc = lane_host_round_trip(who, device, st, on_device ? nullptr : frames, on_device ? 0 : (size_t)n * height * width * 3,
                                        nullptr, scratch_bytes, launch);
    if (rc) return rc;
    for (int i = 0; i < n; i++) {
        out[i].sum_gray = h_acc[4 * i];
        if (strip) {                                         // the strip kernel sums L' = L + 1020
            const long long px = (long long)height * width, sl = (long long)h_acc[4 * i + 1];
            out[i].sum_laplacian = sl - 1020 * px;
            out[i].sum_laplacian_sq = h_acc[4 * i + 2] - 2040ull * (unsigned long long)sl + 1040400ull * (unsigned long long)px;
        } else {
            out[i].sum_laplacian = (int64_t)h_acc[4 * i + 1];
            out[i].sum_laplacian_sq = h_acc[4 * i + 2];
        }
        out[i].green_pixels = h_acc[4 * i + 3];
    }
    return LANE_OK;
}
