// K2: median -> thresholds, Sobel + L1 magnitude + sector NMS + double threshold, hysteresis.
//
// Replaces np.median + the low/high expressions (lane_detector.py:79-81) and cv2.Canny(blurred, low, high)
// (lane_detector.py:83); arithmetic per SURVEY.md A.3/A.4: aperture-3 Sobel with BORDER_REPLICATE,
// mag = |dx|+|dy| with a zero 1-px border, TG22 = 13573 fixed-point sector test, asymmetric >/>= NMS,
// candidates mag > low, strong mag > high, 8-connected closure (unique fixed point, so any
// propagation order is bit-exact).
#include "lane_common.cuh"

namespace {

// ---- thresholds: one thread per frame walks the 256-bin histogram -------------------------
__global__ void k_thresholds(const uint32_t *__restrict__ hist, const uint8_t *__restrict__ lut_low,
                             const uint8_t *__restrict__ lut_high, int4 *__restrict__ thr, int n, long long P)
{
    int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n) return;
    const uint32_t *h = hist + f * 256;
    long long k0 = (P & 1) ? P / 2 : P / 2 - 1, k1 = P / 2;
    long long c = 0;
    int v0 = -1, v1 = -1;
    for (int v = 0; v < 256; v++) {
        c += h[v];
        if (v0 < 0 && c > k0) v0 = v;
        if (v1 < 0 && c > k1) v1 = v;
    }
    int m2 = v0 + v1;
    int lo = lut_low[m2], hi = lut_high[m2];
    if (lo > hi) { int t = lo; lo = hi; hi = t; }
    thr[f] = make_int4(m2, lo, hi, 0);
}

// ---- Sobel + NMS + classification, 32x32 tiles ----------------------------------------------
constexpr int T = 32;

__global__ void __launch_bounds__(256) k_sobel_nms(const uint8_t *__restrict__ blur, const int4 *__restrict__ thr,
                                                   uint8_t *__restrict__ cls, int *__restrict__ seeds,
                                                   int *__restrict__ seed_count, int seed_cap, int H, int W)
{
    __shared__ uint8_t b[T + 4][T + 4];
    __shared__ short sdx[T + 2][T + 2], sdy[T + 2][T + 2];
    __shared__ unsigned short smag[T + 2][T + 2];
    const int tid = threadIdx.x, f = blockIdx.z, x0 = blockIdx.x * T, y0 = blockIdx.y * T;
    const uint8_t *src = blur + (size_t)f * H * W;
    for (int i = tid; i < (T + 4) * (T + 4); i += 256) {
        int ly = i / (T + 4), lx = i - ly * (T + 4);
        int gy = min(max(y0 + ly - 2, 0), H - 1), gx = min(max(x0 + lx - 2, 0), W - 1);   // BORDER_REPLICATE
        b[ly][lx] = src[(size_t)gy * W + gx];
    }
    __syncthreads();
    for (int i = tid; i < (T + 2) * (T + 2); i += 256) {
        int ly = i / (T + 2), lx = i - ly * (T + 2);
        int gy = y0 + ly - 1, gx = x0 + lx - 1;
        int dx = 0, dy = 0, m = 0;
        if (gy >= 0 && gy < H && gx >= 0 && gx < W) {
            const int cy = ly + 1, cx = lx + 1;
            dx = (b[cy - 1][cx + 1] - b[cy - 1][cx - 1]) + 2 * (b[cy][cx + 1] - b[cy][cx - 1]) +
                 (b[cy + 1][cx + 1] - b[cy + 1][cx - 1]);
            dy = (b[cy + 1][cx - 1] - b[cy - 1][cx - 1]) + 2 * (b[cy + 1][cx] - b[cy - 1][cx]) +
                 (b[cy + 1][cx + 1] - b[cy - 1][cx + 1]);
            m = abs(dx) + abs(dy);
        }
        sdx[ly][lx] = (short)dx; sdy[ly][lx] = (short)dy; smag[ly][lx] = (unsigned short)m;
    }
    __syncthreads();
    const int4 t = thr[f];
    const int low = t.y, high = t.z;
    uint8_t *dst = cls + (size_t)f * H * W;
    for (int i = tid; i < T * T; i += 256) {
        int ly = i / T, lx = i - ly * T;
        int gy = y0 + ly, gx = x0 + lx;
        if (gy >= H || gx >= W) continue;
        const int cy = ly + 1, cx = lx + 1;
        int m = smag[cy][cx];
        uint8_t out = 0;
        if (m > low) {
            int dx = sdx[cy][cx], dy = sdy[cy][cx];
            int ax = abs(dx), ay = abs(dy) << 15;
            int tg22x = ax * 13573;
            bool keep;
            if (ay < tg22x) {
                keep = m > smag[cy][cx - 1] && m >= smag[cy][cx + 1];
            } else if (ay > tg22x + (ax << 16)) {
                keep = m > smag[cy - 1][cx] && m >= smag[cy + 1][cx];
            } else {
                int s = ((dx ^ dy) < 0) ? -1 : 1;
                keep = m > smag[cy - 1][cx - s] && m > smag[cy + 1][cx + s];
            }
            if (keep) {
                out = m > high ? 2 : 1;
                if (out == 2) {
                    int pos = atomicAdd(&seed_count[f], 1);
                    if (pos < seed_cap) seeds[(size_t)f * seed_cap + pos] = gy * W + gx;
                }
            }
        }
        dst[(size_t)gy * W + gx] = out;
    }
}

// ---- hysteresis: one CTA per frame, frontier BFS from the strong pixels ------------------------
// Promotion is an atomicOr of bit 1 into the pixel's byte (1 -> 3), so exactly one thread wins each
// weak pixel and pushes it.  If a frontier overflows its buffer the frame falls back to full rescans.
__device__ __forceinline__ bool promote(uint8_t *p)
{
    uintptr_t a = (uintptr_t)p;
    unsigned *w = (unsigned *)(a & ~(uintptr_t)3);
    unsigned sh = (unsigned)(a & 3) * 8;
    unsigned old = atomicOr(w, 2u << sh);
    return ((old >> sh) & 0xFFu) == 1u;
}

__global__ void __launch_bounds__(1024) k_hysteresis(uint8_t *cls, int *bufA, int *bufB,
                                                     const int *__restrict__ seed_count, int cap,
                                                     int *__restrict__ rounds, int H, int W)
{
    __shared__ int s_next, s_over, s_changed;
    const int tid = threadIdx.x, f = blockIdx.x;
    uint8_t *c = cls + (size_t)f * H * W;
    int *cur = bufA + (size_t)f * cap, *nxt = bufB + (size_t)f * cap;
    int ncur = seed_count[f];
    bool overflow = ncur > cap;
    int r = 0;
    while (!overflow && ncur > 0) {
        if (tid == 0) { s_next = 0; s_over = 0; }
        __syncthreads();
        for (int i = tid; i < ncur; i += 1024) {
            int p = cur[i];
            int y = p / W, x = p - y * W;
            for (int oy = -1; oy <= 1; oy++) {
                int yy = y + oy;
                if (yy < 0 || yy >= H) continue;
                for (int ox = -1; ox <= 1; ox++) {
                    int xx = x + ox;
                    if (xx < 0 || xx >= W || (ox == 0 && oy == 0)) continue;
                    uint8_t *q = c + (size_t)yy * W + xx;
                    if (__ldcg(q) == 1 && promote(q)) {
                        int pos = atomicAdd(&s_next, 1);
                        if (pos < cap) nxt[pos] = yy * W + xx; else s_over = 1;
                    }
                }
            }
        }
        __syncthreads();
        ncur = s_next;
        overflow = s_over != 0;
        int *t = cur; cur = nxt; nxt = t;
        r++;
        __syncthreads();
    }
    if (overflow) {
        // Fallback: sweep the whole frame until nothing changes (correct from any intermediate state).
        const int P = H * W;
        for (;;) {
            if (tid == 0) s_changed = 0;
            __syncthreads();
            bool ch = false;
            for (int p = tid; p < P; p += 1024) {
                if (__ldcg(c + p) != 1) continue;
                int y = p / W, x = p - y * W;
                bool nb = false;
                for (int oy = -1; oy <= 1 && !nb; oy++) {
                    int yy = y + oy;
                    if (yy < 0 || yy >= H) continue;
                    for (int ox = -1; ox <= 1; ox++) {
                        int xx = x + ox;
                        if (xx < 0 || xx >= W) continue;
                        if (__ldcg(c + (size_t)yy * W + xx) >= 2) { nb = true; break; }
                    }
                }
                if (nb) { promote(c + p); ch = true; }
            }
            if (ch) s_changed = 1;
            __syncthreads();
            bool again = s_changed != 0;
            r++;
            __syncthreads();
            if (!again) break;
        }
    }
    if (tid == 0) rounds[f] = r;
}

__global__ void k_finalize(uint8_t *__restrict__ cls, int *__restrict__ n_edges, int P)
{
    const int f = blockIdx.y;
    uint8_t *c = cls + (size_t)f * P;
    int cnt = 0;
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < P; p += gridDim.x * blockDim.x) {
        bool e = c[p] >= 2;
        c[p] = e ? 255 : 0;
        cnt += e;
    }
    for (int o = 16; o; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(&n_edges[f], cnt);
}

// ---- ROI mask + ordered compaction: one CTA per frame walks the ROI bounding box row-major -------
__global__ void __launch_bounds__(1024) k_compact(const uint8_t *__restrict__ edges, const uint8_t *__restrict__ roi,
                                                  const int *__restrict__ roi_index, size_t roi_stride,
                                                  uint8_t *__restrict__ pmask, uint32_t *__restrict__ points,
                                                  int *__restrict__ n_points, LaneGeom g)
{
    __shared__ int wpre[32];
    __shared__ int s_total;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, f = blockIdx.x;
    const uint8_t *e = edges + (size_t)f * g.H * g.W;
    if (roi_index) roi += (size_t)roi_index[f] * roi_stride;
    const int area = g.bw * g.bh;
    uint8_t *pm = pmask + (size_t)f * area;
    uint32_t *out = points + (size_t)f * g.max_points;
    int running = 0;   // identical in every thread
    for (int base = 0; base < area; base += 1024) {
        int idx = base + tid;
        bool on = false;
        int x = 0, y = 0;
        if (idx < area) {
            int ry = idx / g.bw;
            y = g.by0 + ry; x = g.bx0 + (idx - ry * g.bw);
            size_t p = (size_t)y * g.W + x;
            on = e[p] != 0 && roi[p] != 0;
            pm[idx] = on ? 1 : 0;
        }
        unsigned bal = __ballot_sync(0xffffffffu, on);
        if (lane == 0) wpre[wid] = __popc(bal);
        __syncthreads();
        if (wid == 0) {
            int v = wpre[lane], inc = v;
            for (int o = 1; o < 32; o <<= 1) {
                int t = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o) inc += t;
            }
            wpre[lane] = inc - v;          // exclusive prefix over warps
            if (lane == 31) s_total = inc;
        }
        __syncthreads();
        if (on) out[running + wpre[wid] + __popc(bal & ((1u << lane) - 1u))] = ((uint32_t)y << 16) | (uint32_t)x;
        running += s_total;
        __syncthreads();
    }
    if (tid == 0) n_points[f] = running;
}

}  // namespace

void launch_thresholds(const uint32_t *hist, const uint8_t *lut_low, const uint8_t *lut_high, int4 *thr,
                       int n, int H, int W, cudaStream_t st, int *launches)
{
    k_thresholds<<<(n + 63) / 64, 64, 0, st>>>(hist, lut_low, lut_high, thr, n, (long long)H * W);
    *launches += 1;
}

void launch_sobel_nms(const uint8_t *blur, const int4 *thr, uint8_t *cls, int *seeds, int *seed_count,
                      int seed_cap, int n, int H, int W, cudaStream_t st, int *launches)
{
    cudaMemsetAsync(seed_count, 0, sizeof(int) * n, st);
    dim3 grid((W + T - 1) / T, (H + T - 1) / T, n);
    k_sobel_nms<<<grid, 256, 0, st>>>(blur, thr, cls, seeds, seed_count, seed_cap, H, W);
    *launches += 1;
}

void launch_hysteresis(uint8_t *cls, int *seeds, int *seeds2, const int *seed_count, int seed_cap,
                       int *rounds, int n, int H, int W, cudaStream_t st, int *launches)
{
    k_hysteresis<<<n, 1024, 0, st>>>(cls, seeds, seeds2, seed_count, seed_cap, rounds, H, W);
    *launches += 1;
}

void launch_finalize_edges(uint8_t *cls_edges, int *n_edges, int n, int H, int W, cudaStream_t st, int *launches)
{
    cudaMemsetAsync(n_edges, 0, sizeof(int) * n, st);
    int P = H * W;
    dim3 grid(min((P + 255) / 256, 296), n);
    k_finalize<<<grid, 256, 0, st>>>(cls_edges, n_edges, P);
    *launches += 1;
}

void launch_compact(const uint8_t *edges, const uint8_t *roi, const int *roi_index, size_t roi_stride, uint8_t *pmask,
                    uint32_t *points, int *n_points, LaneGeom g, int n, cudaStream_t st, int *launches)
{
    k_compact<<<n, 1024, 0, st>>>(edges, roi, roi_index, roi_stride, pmask, points, n_points, g);
    *launches += 1;
}
