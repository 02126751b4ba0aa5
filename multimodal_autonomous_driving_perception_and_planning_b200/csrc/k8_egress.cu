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
#include <stdio.h>

#include <algorithm>
#include <mutex>

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

int efail(int code, const char *what, cudaError_t e = cudaSuccess)
{
    char buf[256];
    snprintf(buf, sizeof buf, "lane_bgr_to_yuv420_batch: %s%s%s", what, e ? ": " : "", e ? cudaGetErrorString(e) : "");
    lane_set_global_error(buf);
    return code;
}

bool device_memory_on(const void *p, int device)
{
    cudaPointerAttributes pa{};
    const bool ok = cudaPointerGetAttributes(&pa, p) == cudaSuccess &&
                    (pa.type == cudaMemoryTypeDevice || pa.type == cudaMemoryTypeManaged) && pa.device == device;
    cudaGetLastError();
    return ok;
}

// Host destinations: chunks of CHUNK output bytes are converted into one of two device scratch slots on the caller's
// stream while the previous chunk is copied out on the copy stream.  One per device, created on first use; the mutex
// serialises host-destination calls, each of which returns with both slots idle.
struct Egress {
    static constexpr size_t CHUNK = (size_t)32 << 20;
    std::mutex mu;
    uint8_t *scratch = nullptr;
    size_t cap = 0;
    cudaStream_t cs = nullptr;
    cudaEvent_t converted[2] = {}, copied[2] = {};

    cudaError_t init()
    {
        if (cs) return cudaSuccess;
        cudaError_t e;
        for (int i = 0; i < 2; i++)
            if ((e = cudaEventCreateWithFlags(&converted[i], cudaEventDisableTiming)) ||
                (e = cudaEventCreateWithFlags(&copied[i], cudaEventDisableTiming)))
                return e;
        return cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking);
    }
    cudaError_t reserve(size_t bytes)
    {
        if (cap >= bytes) return cudaSuccess;
        cudaFree(scratch);
        scratch = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc((void **)&scratch, bytes);
        if (!e) cap = bytes;
        return e;
    }
};

Egress *egress_of(int device)         // one per device, lives until exit
{
    static std::mutex mu;
    static Egress *all[64] = {};
    if (device < 0 || device >= 64) return nullptr;
    std::lock_guard<std::mutex> lk(mu);
    if (!all[device]) all[device] = new Egress();
    return all[device];
}

}  // namespace

extern "C" int lane_bgr_to_yuv420_batch(const uint8_t *src_dev, int format, int n, int height, int width, uint8_t *dst,
                                        int dst_on_device, int device, void *cuda_stream)
{
    if (!src_dev || !dst) return efail(LANE_ERR_INVALID, "null pointer");
    if (format != LANE_INPUT_NV12 && format != LANE_INPUT_I420)
        return efail(LANE_ERR_INVALID, "format must be LANE_INPUT_NV12 or LANE_INPUT_I420");
    if (n < 0 || height < 1 || width < 1) return efail(LANE_ERR_INVALID, "bad sizes (n >= 0, positive height and width)");
    if ((height | width) & 1) return efail(LANE_ERR_INVALID, "YUV 4:2:0 needs even width and height");
    // the kernels grid-stride over 64-bit block indices: the only bound on n is that byte offsets stay below 2^62
    if ((double)n * height * width * 3 > 0x1p62) return efail(LANE_ERR_INVALID, "batch above 2^62 bytes");
    if (n == 0) return LANE_OK;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return efail(LANE_ERR_NO_DEVICE, "no CUDA device visible: this library has no CPU fallback");
    if (device < 0 || device >= ndev) return efail(LANE_ERR_INVALID, "device out of range");
    cudaError_t e;
    if ((e = cudaSetDevice(device))) return efail(LANE_ERR_CUDA, "cudaSetDevice", e);
    if (!device_memory_on(src_dev, device))
        return efail(LANE_ERR_INVALID, "src_dev must be device memory on `device` (host frames: cv2.cvtColor)");
    if (dst_on_device && !device_memory_on(dst, device))
        return efail(LANE_ERR_INVALID, "dst_on_device = 1 needs device memory on `device`");
    cudaStream_t st = (cudaStream_t)cuda_stream;
    if (dst_on_device) {
        launch_bgr_to_yuv420(src_dev, format, dst, n, height, width, st);
        if ((e = cudaGetLastError())) return efail(LANE_ERR_CUDA, "launch", e);
        return LANE_OK;
    }

    Egress *eg = egress_of(device);
    if (!eg) return efail(LANE_ERR_INVALID, "device index above 63");
    std::lock_guard<std::mutex> lk(eg->mu);
    if ((e = eg->init())) return efail(LANE_ERR_CUDA, "copy stream", e);
    const size_t in_frame = (size_t)height * width * 3, out_frame = in_frame / 2;
    const int chunk = (int)std::min<size_t>((size_t)n, std::max<size_t>(1, Egress::CHUNK / out_frame));
    const size_t slot_bytes = (size_t)chunk * out_frame;
    if ((e = eg->reserve(2 * slot_bytes))) return efail(LANE_ERR_CUDA, "scratch allocation", e);
    // pinned / registered destinations and small pageable ones take the DMA directly; large pageable ones the ring
    HostStager *hs = HostStager::pageable(dst, (size_t)n * out_frame) ? lane_host_stager(device) : nullptr;
    const int chunks = (n + chunk - 1) / chunk;
    auto convert = [&](int k) {
        const int slot = k & 1, f0 = k * chunk;
        cudaError_t r;
        if (k >= 2 && (r = cudaStreamWaitEvent(st, eg->copied[slot], 0))) return r;
        launch_bgr_to_yuv420(src_dev + (size_t)f0 * in_frame, format, eg->scratch + slot * slot_bytes,
                             std::min(chunk, n - f0), height, width, st);
        if ((r = cudaGetLastError())) return r;
        return cudaEventRecord(eg->converted[slot], st);
    };
    e = convert(0);
    for (int k = 0; !e && k < chunks; k++) {
        const int slot = k & 1, f0 = k * chunk;
        if (k + 1 < chunks && (e = convert(k + 1))) break;
        if ((e = cudaStreamWaitEvent(eg->cs, eg->converted[slot], 0))) break;
        uint8_t *to = dst + (size_t)f0 * out_frame;
        const uint8_t *from = eg->scratch + slot * slot_bytes;
        const size_t nb = (size_t)std::min(chunk, n - f0) * out_frame;
        e = hs ? hs->d2h(to, from, nb, eg->cs) : cudaMemcpyAsync(to, from, nb, cudaMemcpyDeviceToHost, eg->cs);
        if (!e) e = cudaEventRecord(eg->copied[slot], eg->cs);
    }
    // the copy stream waited for every conversion it copied; after a failure the caller's stream may still hold one
    const cudaError_t s = cudaStreamSynchronize(eg->cs);
    if (e) cudaStreamSynchronize(st);
    if (!e) e = s;
    if (e) return efail(LANE_ERR_CUDA, "conversion to host memory", e);
    return LANE_OK;
}
