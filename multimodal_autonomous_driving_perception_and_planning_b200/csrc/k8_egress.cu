// K8: annotated frames -> a video encoder's input layout, on the device (SURVEY.md 8f rank 3: the step after the
// overlays when annotated video is written).
//
// Every encoder takes 4:2:0 input (libx264 through an FFmpeg pipe with -pix_fmt yuv420p, PyAV, a hardware encoder's
// NV12 surface).  This kernel produces, per frame, exactly cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420) -- or the same
// samples with U and V interleaved (NV12) -- so only 1.5 B/px of the annotated frame has to leave the device.  The
// arithmetic (k0_common.cuh, restated in tests/bgr_yuv420.py) is BT.601 limited range in 20-bit fixed point; U and V come
// from the top-left pixel of each 2x2 block.
//
// HBM-bound: 3 B/px read + 1.5 B/px written.  The vector kernel converts a 2 x 8 pixel block per thread: three 8-byte
// loads per BGR row, one 8-byte Y store per row, then four U and four V bytes (I420) or eight interleaved bytes (NV12).
// The scalar kernel takes one 2x2 block per thread, for any other even width or a misaligned pointer.
#include <algorithm>

#include "host_stage.h"
#include "k0_common.cuh"

namespace {

using namespace k0yuv;

// byte j of the 24 bytes held in w[6]
__device__ __forceinline__ int byte_of(const uint32_t (&w)[6], int j) { return (int)((w[j >> 2] >> (8 * (j & 3))) & 0xFFu); }

__device__ __forceinline__ void load24(const uint8_t *p, uint32_t (&w)[6])
{
    const uint2 *q = reinterpret_cast<const uint2 *>(p);
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const uint2 v = __ldg(q + k);
        w[2 * k] = v.x; w[2 * k + 1] = v.y;
    }
}

// the 8 Y bytes of one row of 8 BGR pixels
__device__ __forceinline__ uint2 row_y(const uint32_t (&w)[6])
{
    uint32_t y[2] = {0u, 0u};
#pragma unroll
    for (int i = 0; i < 8; i++)
        y[i >> 2] |= bgr_y(byte_of(w, 3 * i), byte_of(w, 3 * i + 1), byte_of(w, 3 * i + 2)) << (8 * (i & 3));
    return make_uint2(y[0], y[1]);
}

// W % 8 == 0, 8-byte aligned frames
template <int FMT>
__global__ void __launch_bounds__(256) k8_bgr_to_yuv420_vec(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst,
                                                            int n, int H, int W)
{
    const int bw = W / 8, bh = H / 2;
    const long long total = (long long)n * bh * bw;
    const size_t P = (size_t)H * W, src_frame = P * 3, dst_frame = P * 3 / 2;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int bx = (int)(i % bw);
        const long long q = i / bw;
        const int by = (int)(q % bh), f = (int)(q / bh);
        const uint8_t *s = src + f * src_frame + ((size_t)(2 * by) * W + 8 * bx) * 3;
        uint8_t *d = dst + f * dst_frame;
        uint32_t w[6];
        load24(s + (size_t)W * 3, w);
        *reinterpret_cast<uint2 *>(d + (size_t)(2 * by + 1) * W + 8 * bx) = row_y(w);
        load24(s, w);
        *reinterpret_cast<uint2 *>(d + (size_t)(2 * by) * W + 8 * bx) = row_y(w);
        uint32_t u = 0, v = 0;                       // pixels 0, 2, 4, 6 of the top row
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int b = byte_of(w, 6 * k), g = byte_of(w, 6 * k + 1), r = byte_of(w, 6 * k + 2);
            u |= bgr_u(b, g, r) << (8 * k);
            v |= bgr_v(b, g, r) << (8 * k);
        }
        if constexpr (FMT == LANE_INPUT_NV12) {
            const uint32_t lo = __byte_perm(u, v, 0x5140), hi = __byte_perm(u, v, 0x7362);   // U0 V0 U1 V1 | U2 V2 U3 V3
            *reinterpret_cast<uint2 *>(d + P + (size_t)by * W + 8 * bx) = make_uint2(lo, hi);
        } else {                                     // 4-byte aligned when W % 8 == 0
            const size_t c = P + (size_t)by * (W / 2) + 4 * bx;
            *reinterpret_cast<uint32_t *>(d + c) = u;
            *reinterpret_cast<uint32_t *>(d + c + P / 4) = v;
        }
    }
}

// any even W, H and any alignment: one thread per 2x2 block
template <int FMT>
__global__ void __launch_bounds__(256) k8_bgr_to_yuv420_generic(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst,
                                                                int n, int H, int W)
{
    const int bw = W / 2, bh = H / 2;
    const long long total = (long long)n * bh * bw;
    const size_t P = (size_t)H * W, src_frame = P * 3, dst_frame = P * 3 / 2;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int bx = (int)(i % bw);
        const long long q = i / bw;
        const int by = (int)(q % bh), f = (int)(q / bh);
        const uint8_t *s = src + f * src_frame;
        uint8_t *d = dst + f * dst_frame;
#pragma unroll
        for (int dy = 0; dy < 2; dy++)
#pragma unroll
            for (int dx = 0; dx < 2; dx++) {
                const size_t p = (size_t)(2 * by + dy) * W + 2 * bx + dx;
                d[p] = (uint8_t)bgr_y(__ldg(s + 3 * p), __ldg(s + 3 * p + 1), __ldg(s + 3 * p + 2));
            }
        const size_t p = (size_t)(2 * by) * W + 2 * bx;
        const int b = __ldg(s + 3 * p), g = __ldg(s + 3 * p + 1), r = __ldg(s + 3 * p + 2);
        if constexpr (FMT == LANE_INPUT_NV12) {
            uint8_t *c = d + P + (size_t)by * W + 2 * bx;
            c[0] = (uint8_t)bgr_u(b, g, r); c[1] = (uint8_t)bgr_v(b, g, r);
        } else {
            const size_t c = P + (size_t)by * (W / 2) + bx;
            d[c] = (uint8_t)bgr_u(b, g, r); d[c + P / 4] = (uint8_t)bgr_v(b, g, r);
        }
    }
}

template <int FMT>
void launch_fmt(const uint8_t *src, uint8_t *dst, int n, int H, int W, cudaStream_t st)
{
    const int sms = lane_sm_count();
    if (W % 8 == 0 && (((uintptr_t)src | (uintptr_t)dst) % 8) == 0) {
        const long long total = (long long)n * (H / 2) * (W / 8);
        const int blocks = (int)std::min<long long>((total + 255) / 256, (long long)sms * 16);
        k8_bgr_to_yuv420_vec<FMT><<<std::max(blocks, 1), 256, 0, st>>>(src, dst, n, H, W);
    } else {
        const long long total = (long long)n * (H / 2) * (W / 2);
        const int blocks = (int)std::min<long long>((total + 255) / 256, (long long)sms * 16);
        k8_bgr_to_yuv420_generic<FMT><<<std::max(blocks, 1), 256, 0, st>>>(src, dst, n, H, W);
    }
}

void launch_bgr_to_yuv420(const uint8_t *src, int format, uint8_t *dst, int n, int H, int W, cudaStream_t st)
{
    if (format == LANE_INPUT_I420)
        launch_fmt<LANE_INPUT_I420>(src, dst, n, H, W, st);
    else
        launch_fmt<LANE_INPUT_NV12>(src, dst, n, H, W, st);
}

bool device_memory_on(const void *p, int device)
{
    cudaPointerAttributes pa{};
    const bool ok = cudaPointerGetAttributes(&pa, p) == cudaSuccess &&
                    (pa.type == cudaMemoryTypeDevice || pa.type == cudaMemoryTypeManaged) && pa.device == device;
    cudaGetLastError();
    return ok;
}

}  // namespace

extern "C" int lane_bgr_to_yuv420_batch(const uint8_t *src_dev, int format, int n, int height, int width, uint8_t *dst,
                                        int dst_on_device, int device, void *cuda_stream)
{
    constexpr const char *who = "lane_bgr_to_yuv420_batch";
    if (!src_dev || !dst) return lane_api_fail(LANE_ERR_INVALID, who, "null pointer");
    if (format != LANE_INPUT_NV12 && format != LANE_INPUT_I420)
        return lane_api_fail(LANE_ERR_INVALID, who, "format must be LANE_INPUT_NV12 or LANE_INPUT_I420");
    if (n < 0 || height < 1 || width < 1) return lane_api_fail(LANE_ERR_INVALID, who, "bad sizes (n >= 0, positive height and width)");
    if ((height | width) & 1) return lane_api_fail(LANE_ERR_INVALID, who, "YUV 4:2:0 needs even width and height");
    // the kernels grid-stride over 64-bit block indices: the only bound on n is that byte offsets stay below 2^62
    if ((double)n * height * width * 3 > 0x1p62) return lane_api_fail(LANE_ERR_INVALID, who, "batch above 2^62 bytes");
    if (n == 0) return LANE_OK;
    if (int rc = lane_api_device(who, device)) return rc;
    if (!device_memory_on(src_dev, device))
        return lane_api_fail(LANE_ERR_INVALID, who, "src_dev must be device memory on `device` (host frames: cv2.cvtColor)");
    if (dst_on_device && !device_memory_on(dst, device))
        return lane_api_fail(LANE_ERR_INVALID, who, "dst_on_device = 1 needs device memory on `device`");
    cudaStream_t st = (cudaStream_t)cuda_stream;
    cudaError_t e;
    if (dst_on_device) {
        launch_bgr_to_yuv420(src_dev, format, dst, n, height, width, st);
        if ((e = cudaGetLastError())) return lane_api_fail(LANE_ERR_CUDA, who, "launch", e);
        return LANE_OK;
    }

    // Host destinations: chunks of CHUNK output bytes are converted into one of two slots of the device's scratch on the
    // caller's stream while the previous chunk is copied out on the device's copy stream.
    constexpr size_t CHUNK = (size_t)32 << 20;
    LaneDeviceHost &h = lane_device_host(device);
    std::lock_guard<std::mutex> lk(h.mu);
    if ((e = h.init_copy_stream())) return lane_api_fail(LANE_ERR_CUDA, who, "copy stream", e);
    const size_t in_frame = (size_t)height * width * 3, out_frame = in_frame / 2;
    const int chunk = (int)std::min<size_t>((size_t)n, std::max<size_t>(1, CHUNK / out_frame));
    const size_t slot_bytes = (size_t)chunk * out_frame;
    if ((e = h.scratch.grow(2 * slot_bytes))) return lane_api_fail(LANE_ERR_CUDA, who, "scratch allocation", e);
    // pinned / registered destinations and small pageable ones take the DMA directly; large pageable ones the ring
    const bool staged = HostStager::pageable(dst, (size_t)n * out_frame);
    const int chunks = (n + chunk - 1) / chunk;
    auto convert = [&](int k) {
        const int slot = k & 1, f0 = k * chunk;
        cudaError_t r;
        if (k >= 2 && (r = cudaStreamWaitEvent(st, h.copied[slot], 0))) return r;
        launch_bgr_to_yuv420(src_dev + (size_t)f0 * in_frame, format, h.scratch + slot * slot_bytes,
                             std::min(chunk, n - f0), height, width, st);
        if ((r = cudaGetLastError())) return r;
        return cudaEventRecord(h.converted[slot], st);
    };
    e = convert(0);
    for (int k = 0; !e && k < chunks; k++) {
        const int slot = k & 1, f0 = k * chunk;
        if (k + 1 < chunks && (e = convert(k + 1))) break;
        if ((e = cudaStreamWaitEvent(h.copy_st, h.converted[slot], 0))) break;
        uint8_t *to = dst + (size_t)f0 * out_frame;
        const uint8_t *from = h.scratch + slot * slot_bytes;
        const size_t nb = (size_t)std::min(chunk, n - f0) * out_frame;
        e = staged ? h.stager.d2h(to, from, nb, h.copy_st) : cudaMemcpyAsync(to, from, nb, cudaMemcpyDeviceToHost, h.copy_st);
        if (!e) e = cudaEventRecord(h.copied[slot], h.copy_st);
    }
    // the copy stream waited for every conversion it copied; after a failure the caller's stream may still hold one
    const cudaError_t s = cudaStreamSynchronize(h.copy_st);
    if (e) cudaStreamSynchronize(st);
    if (!e) e = s;
    if (e) return lane_api_fail(LANE_ERR_CUDA, who, "conversion to host memory", e);
    return LANE_OK;
}
