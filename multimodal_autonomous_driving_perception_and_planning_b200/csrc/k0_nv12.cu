// K0b: frame ingest, NV12 -> BGR (SURVEY.md 8f rank 1, second half).
//
// Frames enter the reference through VideoDataLoader.read_frame / read_frame_at
// (/root/reference/data/loaders/video_loader.py:96-131), i.e. out of a video decoder.  A hardware decoder hands out
// NV12 (Y plane + half-resolution interleaved UV plane, 1.5 B/px); the BGR frame the lane path consumes is what
// cv2.cvtColor(nv12, cv2.COLOR_YUV2BGR_NV12) makes of it.  Doing that conversion on the device halves the bytes that
// cross PCIe per frame, which is what bounds the end-to-end rate.  Bit-exact against cv2 (oracle/nv12.py restates the
// arithmetic: ITU-R BT.601 limited range, 20-bit fixed point, arithmetic shift, saturation).
//
// I420 (what software decoders hand out: U and V as separate quarter planes) carries the same samples and converts with
// the same arithmetic; the kernels are templated on the chroma addressing (k0_common.cuh).
//
// HBM-bound: 1.5 B/px read + 3 B/px written.  A thread converts a 2 x 8 pixel block: one 8-byte load per luma row,
// one 8-byte load of the four (U, V) pairs the block shares, three 8-byte stores per output row; a warp covers
// 256 px of two rows, so every access is a full, aligned segment.
//
// K0f at the source size: packed YUV 4:2:2 (UYVY / YUYV, 2 B/px) -> BGR with the same arithmetic.  Nothing is shared
// between rows, so a batch of dense frames is one run of pixel pairs: a thread converts 8 pixels with one 16-byte load,
// PRMT splits it into the 8 Y bytes and the 4 (U, V) pairs, and row8 makes the 24 BGR bytes (three 8-byte stores).
// 2 B/px read + 3 B/px written.
#include <algorithm>

#include "k0_common.cuh"

namespace {

using namespace k0yuv;

// 8 luma bytes of one row + the four chroma terms -> 24 BGR bytes (six words)
__device__ __forceinline__ void row8(uint2 yy, const UV (&t)[4], uint32_t (&o)[6])
{
    uint32_t b[8], g[8], r[8];
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const int yv = (int)(((i < 4 ? yy.x : yy.y) >> (8 * (i & 3))) & 0xFFu);
        px(yv, t[i >> 1], b[i], g[i], r[i]);
    }
    // B0 G0 R0 B1 | G1 R1 B2 G2 | R2 B3 G3 R3 | ...
#pragma unroll
    for (int h = 0; h < 2; h++) {
        const int k = 4 * h;
        o[3 * h + 0] = b[k] | (g[k] << 8) | (r[k] << 16) | (b[k + 1] << 24);
        o[3 * h + 1] = g[k + 1] | (r[k + 1] << 8) | (b[k + 2] << 16) | (g[k + 2] << 24);
        o[3 * h + 2] = r[k + 2] | (b[k + 3] << 8) | (g[k + 3] << 16) | (r[k + 3] << 24);
    }
}

// W % 8 == 0, 8-byte aligned planes
template <int FMT>
__global__ void __launch_bounds__(256) k0_nv12_vec(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, int n, int H,
                                                   int W)
{
    const int bw = W / 8, bh = H / 2;
    const long long total = (long long)n * bh * bw;
    const size_t src_frame = (size_t)H * W * 3 / 2, dst_frame = (size_t)H * W * 3;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int bx = (int)(i % bw);
        const long long q = i / bw;
        const int by = (int)(q % bh), f = (int)(q / bh);
        const uint8_t *s = src + f * src_frame;
        const uint2 y0 = __ldg(reinterpret_cast<const uint2 *>(s + (size_t)(2 * by) * W + 8 * bx));
        const uint2 y1 = __ldg(reinterpret_cast<const uint2 *>(s + (size_t)(2 * by + 1) * W + 8 * bx));
        UV t[4];
        if constexpr (FMT == LANE_INPUT_NV12) {
            const uint2 uv = __ldg(reinterpret_cast<const uint2 *>(s + (size_t)(H + by) * W + 8 * bx));
            t[0] = uv_terms((int)(uv.x & 0xFFu), (int)((uv.x >> 8) & 0xFFu));
            t[1] = uv_terms((int)((uv.x >> 16) & 0xFFu), (int)(uv.x >> 24));
            t[2] = uv_terms((int)(uv.y & 0xFFu), (int)((uv.y >> 8) & 0xFFu));
            t[3] = uv_terms((int)((uv.y >> 16) & 0xFFu), (int)(uv.y >> 24));
        } else {                       // four U bytes, four V bytes: 4-byte aligned when W % 8 == 0
            const size_t P = (size_t)H * W, q = P + (size_t)by * (W / 2) + 4 * bx;
            const uint32_t u = __ldg(reinterpret_cast<const uint32_t *>(s + q));
            const uint32_t v = __ldg(reinterpret_cast<const uint32_t *>(s + q + P / 4));
#pragma unroll
            for (int i = 0; i < 4; i++) t[i] = uv_terms((int)((u >> (8 * i)) & 0xFFu), (int)((v >> (8 * i)) & 0xFFu));
        }
        uint32_t o[6];
        uint8_t *d = dst + f * dst_frame + ((size_t)(2 * by) * W + 8 * bx) * 3;
        row8(y0, t, o);
        uint2 *d0 = reinterpret_cast<uint2 *>(d);
        d0[0] = make_uint2(o[0], o[1]); d0[1] = make_uint2(o[2], o[3]); d0[2] = make_uint2(o[4], o[5]);
        row8(y1, t, o);
        uint2 *d1 = reinterpret_cast<uint2 *>(d + (size_t)W * 3);
        d1[0] = make_uint2(o[0], o[1]); d1[1] = make_uint2(o[2], o[3]); d1[2] = make_uint2(o[4], o[5]);
    }
}

// any even W, H: one thread per 2x2 block
template <int FMT>
__global__ void __launch_bounds__(256) k0_nv12_generic(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, int n, int H,
                                                       int W)
{
    const int bw = W / 2, bh = H / 2;
    const long long total = (long long)n * bh * bw;
    const size_t src_frame = (size_t)H * W * 3 / 2, dst_frame = (size_t)H * W * 3;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int bx = (int)(i % bw);
        const long long q = i / bw;
        const int by = (int)(q % bh), f = (int)(q / bh);
        const uint8_t *s = src + f * src_frame;
        const UV t = chroma<FMT>(s, H, W, by, bx);
#pragma unroll
        for (int dy = 0; dy < 2; dy++)
#pragma unroll
            for (int dx = 0; dx < 2; dx++) {
                const size_t p = (size_t)(2 * by + dy) * W + 2 * bx + dx;
                uint32_t b, g, r;
                px(s[p], t, b, g, r);
                uint8_t *d = dst + f * dst_frame + p * 3;
                d[0] = (uint8_t)b; d[1] = (uint8_t)g; d[2] = (uint8_t)r;
            }
    }
}

// PRMT selectors of a 16-byte 4:2:2 group of 8 pixels (words w0..w3, little-endian) by Y0 offset YO: the Y bytes of
// words (w0, w1) / (w2, w3), and the (U, V) bytes of one word pair as U0 V0 U1 V1.
template <int YO> constexpr uint32_t Y_SEL = YO ? 0x7531u : 0x6420u;
template <int YO> constexpr uint32_t UV_SEL = YO ? 0x6420u : 0x7531u;

// 8 pixels of one 4:2:2 row (16 source bytes) -> 24 BGR bytes at d (8-byte aligned)
template <int YO>
__device__ __forceinline__ void yuv422_8px(uint4 w, uint2 *__restrict__ d)
{
    const uint2 yy = make_uint2(__byte_perm(w.x, w.y, Y_SEL<YO>), __byte_perm(w.z, w.w, Y_SEL<YO>));
    const uint32_t uv01 = __byte_perm(w.x, w.y, UV_SEL<YO>), uv23 = __byte_perm(w.z, w.w, UV_SEL<YO>);
    UV t[4];
    t[0] = uv_terms((int)(uv01 & 0xFFu), (int)((uv01 >> 8) & 0xFFu));
    t[1] = uv_terms((int)((uv01 >> 16) & 0xFFu), (int)(uv01 >> 24));
    t[2] = uv_terms((int)(uv23 & 0xFFu), (int)((uv23 >> 8) & 0xFFu));
    t[3] = uv_terms((int)((uv23 >> 16) & 0xFFu), (int)(uv23 >> 24));
    uint32_t o[6];
    row8(yy, t, o);
    d[0] = make_uint2(o[0], o[1]); d[1] = make_uint2(o[2], o[3]); d[2] = make_uint2(o[4], o[5]);
}

// W % 8 == 0, 16-byte aligned source, 8-byte aligned destination: one thread = 8 pixels of one row
template <int YO>
__global__ void __launch_bounds__(256) k0_yuv422_vec(const uint4 *__restrict__ src, uint2 *__restrict__ dst, long long groups)
{
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < groups; i += (long long)gridDim.x * blockDim.x)
        yuv422_8px<YO>(__ldg(src + i), dst + 3 * i);
}

// any even W and alignment: one thread per pixel pair (4 source bytes, 6 destination bytes)
__global__ void __launch_bounds__(256) k0_yuv422_generic(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, int yo,
                                                         long long pairs)
{
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < pairs; i += (long long)gridDim.x * blockDim.x) {
        const uint8_t *g = src + 4 * i;
        const UV t = uv_terms(__ldg(g + 1 - yo), __ldg(g + 3 - yo));
        uint8_t *d = dst + 6 * i;
#pragma unroll
        for (int k = 0; k < 2; k++) {
            uint32_t b, gr, r;
            px(__ldg(g + yo + 2 * k), t, b, gr, r);
            d[3 * k] = (uint8_t)b; d[3 * k + 1] = (uint8_t)gr; d[3 * k + 2] = (uint8_t)r;
        }
    }
}

int grid_for(long long threads)
{
    return (int)std::max<long long>(1, std::min<long long>((threads + 255) / 256, (long long)lane_sm_count() * 16));
}

template <int FMT>
void launch_fmt(const uint8_t *src, uint8_t *dst, int n, int H, int W, cudaStream_t st)
{
    const int sms = lane_sm_count();
    if (W % 8 == 0 && (((uintptr_t)src | (uintptr_t)dst) % 8) == 0) {
        const long long total = (long long)n * (H / 2) * (W / 8);
        const int blocks = (int)std::min<long long>((total + 255) / 256, (long long)sms * 16);
        k0_nv12_vec<FMT><<<std::max(blocks, 1), 256, 0, st>>>(src, dst, n, H, W);
    } else {
        const long long total = (long long)n * (H / 2) * (W / 2);
        const int blocks = (int)std::min<long long>((total + 255) / 256, (long long)sms * 16);
        k0_nv12_generic<FMT><<<std::max(blocks, 1), 256, 0, st>>>(src, dst, n, H, W);
    }
}

}  // namespace

// YUV 4:2:0 (LANE_INPUT_NV12 / LANE_INPUT_I420) -> BGR at the same size; device pointers, enqueued on st
void launch_yuv420_to_bgr(const uint8_t *src, int format, uint8_t *dst, int n, int H, int W, cudaStream_t st)
{
    if (format == LANE_INPUT_I420)
        launch_fmt<LANE_INPUT_I420>(src, dst, n, H, W, st);
    else
        launch_fmt<LANE_INPUT_NV12>(src, dst, n, H, W, st);
}

// packed YUV 4:2:2 (LANE_INPUT_UYVY / LANE_INPUT_YUYV) -> BGR at the same size (W even); device pointers, enqueued on st
void launch_yuv422_to_bgr(const uint8_t *src, int format, uint8_t *dst, int n, int H, int W, cudaStream_t st)
{
    const long long px = (long long)n * H * W;
    if (W % 8 == 0 && (uintptr_t)src % 16 == 0 && (uintptr_t)dst % 8 == 0) {
        const auto *s = reinterpret_cast<const uint4 *>(src);
        auto *d = reinterpret_cast<uint2 *>(dst);
        if (format == LANE_INPUT_UYVY)
            k0_yuv422_vec<1><<<grid_for(px / 8), 256, 0, st>>>(s, d, px / 8);
        else
            k0_yuv422_vec<0><<<grid_for(px / 8), 256, 0, st>>>(s, d, px / 8);
    } else {
        k0_yuv422_generic<<<grid_for(px / 2), 256, 0, st>>>(src, dst, lane_yuv422_y0(format), px / 2);
    }
}
