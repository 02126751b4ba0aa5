// Shared pieces of the frame-ingest kernels (K0): the YUV 4:2:0 -> BGR arithmetic of k0_nv12.cu / k0_ingest.cu, its
// inverse for the egress kernel (k8_egress.cu), the packed 4:2:2 addressing and the Bayer demosaic of k0_ingest.cu and
// the INTER_LINEAR tap tables and vertical step of k0_resize.cu.
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

// The per-thread pixel work of the resize kernels (k0_resize, k0_ingest_resize, k0_rig_ingest): one
// thread makes PX consecutive destination pixels dx0 .. dx0+PX-1 of destination row dy (columns past dw repeat the last
// one and are not stored).  yy / b: the row's yofs / beta entries.
//
// k0_resize's arithmetic on CN interleaved uint8 channels: r0 / r1 are the two source rows.
template <int CN, int PX>
__device__ __forceinline__ void k0_resize_px(const uint8_t *__restrict__ r0, const uint8_t *__restrict__ r1,
                                             const int *__restrict__ xofs, const short2 *__restrict__ alpha, short2 b, int sw,
                                             int dx0, int dw, uint8_t (&px)[PX * CN])
{
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
}

// The same resize of the BGR frame cv2.cvtColor makes of YUV 4:2:0 frame `s` (sh x sw luma, layout FMT): the two source
// rows x two source columns of every tap are converted on the fly, the converted frame is never stored.
template <int FMT, int PX>
__device__ __forceinline__ void k0_yuv420_resize_px(const uint8_t *__restrict__ s, int sh, int sw, int2 yy, short2 b,
                                                    const int *__restrict__ xofs, const short2 *__restrict__ alpha, int dx0,
                                                    int dw, uint8_t (&o)[PX * 3])
{
    using namespace k0yuv;
    const uint8_t *l0 = s + (size_t)yy.x * sw, *l1 = s + (size_t)yy.y * sw;
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
}

// ---- packed YUV 4:2:2 -> BGR, bit-exact with cv2.cvtColor(f, COLOR_YUV2BGR_UYVY / COLOR_YUV2BGR_YUY2) (oracle/yuv422.py)
// The per-pixel arithmetic of NV12 (k0yuv::px / uv_terms); each horizontal pixel pair shares the (U, V) of its 4-byte
// group, nothing is shared vertically.  Within a group UYVY stores U Y0 V Y1 and YUYV Y0 U Y1 V: with yo the offset of
// Y0 (1 for UYVY, 0 for YUYV), Y of pixel x is byte 2x + yo of its row, U byte (x & ~1) * 2 + 1 - yo and V the byte two
// after U.
__host__ __device__ constexpr bool lane_input_yuv422(int format)
{
    return format == LANE_INPUT_UYVY || format == LANE_INPUT_YUYV;
}

// yo of a LANE_INPUT_UYVY / YUYV layout: the byte offset of Y0 in each 4-byte group.
__host__ __device__ constexpr int lane_yuv422_y0(int format) { return format == LANE_INPUT_UYVY ? 1 : 0; }

// BGR of pixel x of a 4:2:2 row whose Y bytes are ly[2x] and whose pair (U, V) bytes are lc[(x & ~1) * 2] and two after.
__device__ __forceinline__ void k0_yuv422_px(const uint8_t *__restrict__ ly, const uint8_t *__restrict__ lc, int x,
                                             uint32_t (&p)[3])
{
    const uint8_t *c = lc + (x & ~1) * 2;
    k0yuv::px(__ldg(ly + 2 * x), k0yuv::uv_terms(__ldg(c), __ldg(c + 2)), p[0], p[1], p[2]);
}

// The same resize of the BGR frame cv2.cvtColor makes of packed 4:2:2 frame `s` (sw pixels wide, Y0 at byte offset yo
// of each group): the two source rows x two source columns of every tap are converted on the fly, the converted frame
// is never stored.  At identity taps this is cv2.cvtColor's frame itself.
template <int PX>
__device__ __forceinline__ void k0_yuv422_resize_px(const uint8_t *__restrict__ s, int sw, int yo, int2 yy, short2 b,
                                                    const int *__restrict__ xofs, const short2 *__restrict__ alpha, int dx0,
                                                    int dw, uint8_t (&o)[PX * 3])
{
    const uint8_t *l0 = s + (size_t)yy.x * sw * 2, *l1 = s + (size_t)yy.y * sw * 2;
#pragma unroll
    for (int k = 0; k < PX; k++) {
        const int dx = min(dx0 + k, dw - 1);
        const int x0 = __ldg(xofs + dx), x1 = min(x0 + 1, sw - 1);
        const short2 a = __ldg(alpha + dx);
        uint32_t p00[3], p01[3], p10[3], p11[3];     // BGR of (row y0 | y1) x (column x0 | x1)
        k0_yuv422_px(l0 + yo, l0 + 1 - yo, x0, p00);
        k0_yuv422_px(l0 + yo, l0 + 1 - yo, x1, p01);
        k0_yuv422_px(l1 + yo, l1 + 1 - yo, x0, p10);
        k0_yuv422_px(l1 + yo, l1 + 1 - yo, x1, p11);
#pragma unroll
        for (int c = 0; c < 3; c++) {
            const int h0 = (int)p00[c] * a.x + (int)p01[c] * a.y;
            const int h1 = (int)p10[c] * a.x + (int)p11[c] * a.y;
            o[k * 3 + c] = (uint8_t)k0_vmix(h0, h1, b.x, b.y);
        }
    }
}

// ---- raw Bayer -> BGR, bit-exact with cv2.cvtColor(f, COLOR_Bayer{RGGB,BGGR,GRBG,GBRG}2BGR) (oracle/bayer.py) -------
// The bilinear demosaic.  Pixel (y, x) of an H x W mosaic (H, W >= 3) is the interior formula at (clamp(y, 1, H-2),
// clamp(x, 1, W-2)): its own colour is the raw value; at an R or B site G = (4 neighbours + 2) >> 2 and the other chroma
// = (4 diagonals + 2) >> 2; at a G site the colour of the horizontal neighbours = (left + right + 1) >> 1 and that of
// the vertical ones = (up + down + 1) >> 1.  The four patterns are one RGGB mosaic read at a phase (py, px).
__host__ __device__ constexpr bool lane_input_bayer(int format)
{
    return format >= LANE_INPUT_BAYER_RGGB && format <= LANE_INPUT_BAYER_GBRG;
}

// (py, px) of a LANE_INPUT_BAYER_* layout as bits 1 and 0: RGGB 0, GRBG 1, GBRG 2, BGGR 3.
__host__ __device__ constexpr int lane_bayer_phase(int format)
{
    return format == LANE_INPUT_BAYER_RGGB ? 0 : format == LANE_INPUT_BAYER_GRBG ? 1 : format == LANE_INPUT_BAYER_GBRG ? 2 : 3;
}

// ---- the LANE_INPUT_* layouts: what the host checks, byte counts and kernel choices of every ingest path ask ---------
// (loaders/frame_layout.py is the Python side's table.)
__host__ __device__ constexpr bool lane_input_yuv420(int format)
{
    return format == LANE_INPUT_NV12 || format == LANE_INPUT_I420;
}

// Bytes of n dense h x w frames: 3 B/px BGR, 1.5 B/px YUV 4:2:0, 1 B/px Bayer, 2 B/px YUV 4:2:2.
__host__ __device__ constexpr size_t lane_input_frame_bytes(int format, int h, int w, size_t n = 1)
{
    const size_t px = n * h * w;
    return format == LANE_INPUT_BGR ? px * 3 : lane_input_bayer(format) ? px : lane_input_yuv422(format) ? px * 2 : px * 3 / 2;
}

// Why h x w frames (h, w >= 1) of `format` cannot be taken, or null: an unknown layout, odd 4:2:0 sizes (the chroma
// blocks are 2 x 2), Bayer frames below 3 x 3 (cv2.cvtColor makes an all-zero frame of them), odd 4:2:2 widths.
inline const char *lane_input_refusal(int format, int h, int w)
{
    if (lane_input_yuv420(format)) return (h | w) & 1 ? "YUV 4:2:0 needs even width and height" : nullptr;
    if (lane_input_bayer(format)) return h < 3 || w < 3 ? "a Bayer frame needs at least 3 rows and 3 columns" : nullptr;
    if (lane_input_yuv422(format)) return w & 1 ? "YUV 4:2:2 needs an even width" : nullptr;
    return format == LANE_INPUT_BGR ? nullptr : "unknown input format";
}

// Whether sh x sw frames of `format` become dh x dw BGR on a resizing grid (one block row per destination row, one z
// per frame: dh and the batch up to 65535): at every other size, and Bayer frames at every size (their demosaic is that
// kernel on identity taps).  Otherwise BGR needs no kernel and YUV takes k0_nv12's conversion.
__host__ __device__ constexpr bool lane_input_resizes(int format, int sh, int sw, int dh, int dw)
{
    return sh != dh || sw != dw || lane_input_bayer(format);
}

namespace k0bayer {

// BGR of the centre of the 3x3 window of w at column J (columns J-1..J+1), whose site is at parity (ry, rx) of the RGGB
// mosaic.
template <int J>
__device__ __forceinline__ void px(const int (&w)[3][4], int ry, int rx, int &b, int &g, int &r)
{
    const int own = w[1][J], h = w[1][J - 1] + w[1][J + 1], v = w[0][J] + w[2][J];
    const int d = w[0][J - 1] + w[0][J + 1] + w[2][J - 1] + w[2][J + 1];
    const bool chroma_site = ry == rx;                       // R (0, 0) or B (1, 1); else G
    const int near = chroma_site ? own : (h + 1) >> 1;      // R on a red row, B on a blue row
    const int far = chroma_site ? (d + 2) >> 2 : (v + 1) >> 1;
    g = chroma_site ? (h + v + 2) >> 2 : own;
    r = ry ? far : near;
    b = ry ? near : far;
}

// k0_resize's horizontal step on the demosaiced row cy (clamped, 1 <= cy <= sh-2; site parity ry): the two source
// columns of the tap are the clamped centres cx0 and cx0 + ddx (ddx 0 or 1), demosaiced from the 3x4 raw window at
// rows cy-1..cy+1, columns cx0-1..cx0+2.  `up` points at row cy-1.
__device__ __forceinline__ void hmix(const uint8_t *__restrict__ up, int sw, int cx0, int ddx, int ry, int rx, short2 a,
                                     int (&h)[3])
{
    const int x3 = min(cx0 + 2, sw - 1);                    // columns cx0-1 .. cx0+1 are inside the row
    int w[3][4];
#pragma unroll
    for (int i = 0; i < 3; i++) {
        const uint8_t *r = up + i * sw;
        w[i][0] = __ldg(r + cx0 - 1); w[i][1] = __ldg(r + cx0); w[i][2] = __ldg(r + cx0 + 1); w[i][3] = __ldg(r + x3);
    }
    int p0[3], p1[3];
    px<1>(w, ry, rx, p0[0], p0[1], p0[2]);
    px<2>(w, ry, rx ^ 1, p1[0], p1[1], p1[2]);
#pragma unroll
    for (int c = 0; c < 3; c++) h[c] = p0[c] * a.x + (ddx ? p1[c] : p0[c]) * a.y;
}

}  // namespace k0bayer

// The same resize of the BGR frame cv2.cvtColor makes of Bayer mosaic `s` (sh x sw, sh and sw >= 3, phase as
// lane_bayer_phase): the two source rows x two source columns of every tap are demosaiced on the fly from their raw
// neighbourhood (the clamped centres of y1 / x1 are those of y0 / x0 or one further), the demosaiced frame is never
// stored.  At identity taps this is cv2.cvtColor's frame itself.  dy below is uniform over a destination row.
template <int PX>
__device__ __forceinline__ void k0_bayer_resize_px(const uint8_t *__restrict__ s, int sh, int sw, int phase, int2 yy,
                                                   short2 b, const int *__restrict__ xofs, const short2 *__restrict__ alpha,
                                                   int dx0, int dw, uint8_t (&o)[PX * 3])
{
    const int cy0 = min(max(yy.x, 1), sh - 2), dy = min(max(yy.y, 1), sh - 2) - cy0;        // dy: 0 or 1
    const uint8_t *up = s + (size_t)(cy0 - 1) * sw;
    const int ry = (cy0 + (phase >> 1)) & 1;
#pragma unroll
    for (int k = 0; k < PX; k++) {
        const int dx = min(dx0 + k, dw - 1);
        const int x0 = __ldg(xofs + dx), x1 = min(x0 + 1, sw - 1);
        const short2 a = __ldg(alpha + dx);
        const int cx0 = min(max(x0, 1), sw - 2), ddx = min(max(x1, 1), sw - 2) - cx0;
        const int rx = (cx0 + phase) & 1;
        int h0[3], h1[3];
        k0bayer::hmix(up, sw, cx0, ddx, ry, rx, a, h0);
        if (dy) {
            k0bayer::hmix(up + sw, sw, cx0, ddx, ry ^ 1, rx, a, h1);
        } else {
#pragma unroll
            for (int c = 0; c < 3; c++) h1[c] = h0[c];
        }
#pragma unroll
        for (int c = 0; c < 3; c++) o[k * 3 + c] = (uint8_t)k0_vmix(h0[c], h1[c], b.x, b.y);
    }
}

// Stores one thread's pixels at `out` (destination pixel dx0): packed 4-byte stores when the PX pixels are all inside
// the row and `out` is aligned, byte stores otherwise.
template <int CN, int PX>
__device__ __forceinline__ void k0_store_px(uint8_t *__restrict__ out, const uint8_t (&px)[PX * CN], int dx0, int dw)
{
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

// Tables for the current device (cached; the first call of a geometry allocates and uploads them synchronously).
cudaError_t lane_resize_taps(int sh, int sw, int dh, int dw, ResizeTaps *t);
// k0_resize over n dense frames of `channels` (1 or 3) uint8 planes; device pointers, enqueued on st, no checks.
void launch_resize(const uint8_t *src, uint8_t *dst, int n, int channels, int sh, int sw, int dh, int dw,
                   const ResizeTaps &t, cudaStream_t st);

// k0_nv12: YUV 4:2:0 -> BGR at the source size
void launch_yuv420_to_bgr(const uint8_t *src, int format, uint8_t *dst, int n, int H, int W, cudaStream_t st);
// k0_nv12: packed YUV 4:2:2 (LANE_INPUT_UYVY / YUYV) -> BGR at the source size (W even)
void launch_yuv422_to_bgr(const uint8_t *src, int format, uint8_t *dst, int n, int H, int W, cudaStream_t st);

// ---- ingest: any LANE_INPUT_* layout at any size -> BGR at dh x dw --------------------------------------------------
// NV12 / I420 / UYVY / YUYV at the destination size: k0_nv12's conversion kernels; at another size: the fused
// conversion + resize kernel (k0_ingest_resize); Bayer at any size: the fused demosaic + resize kernel (identity taps at
// its own size); BGR at another size: k0_resize.  BGR at its own size needs no kernel and is not taken.  Device pointers,
// enqueued on st; the caller has validated the sizes (lane_input_refusal) and the grid (lane_input_resizes).
cudaError_t launch_ingest(const uint8_t *src, int format, int n, int sh, int sw, uint8_t *dst, int dh, int dw,
                          cudaStream_t st);

// ---- rig ingest: a batch whose frames each have their own layout and size -> BGR at dh x dw, one launch ------------
// Descriptor of one source frame (device memory, dense); the tap tables are lane_resize_taps' cached ones.
struct RigFrame {
    const uint8_t *src;
    int format, sh, sw;                // LANE_INPUT_*, at a size lane_input_refusal takes
    const int *xofs;
    const short2 *alpha;
    const int2 *yofs;
    const short2 *beta;
};
// The descriptor of frame `src` for a destination of dh x dw (looks up / builds the geometry's tap tables).
cudaError_t rig_frame(const uint8_t *src, int format, int sh, int sw, int dh, int dw, RigFrame *d);
// k0_rig_ingest over n frames: frames_dev = device RigFrame[n], dst = [n][dh][dw][3]; enqueued on st, no checks
// (n and dh up to 65535).
void launch_rig_ingest(const RigFrame *frames_dev, int n, uint8_t *dst, int dh, int dw, cudaStream_t st);
