// K7: batched cv2-exact rasteriser (SURVEY.md 8f ranks 3 and 4: the step right after the lane path, and its input fixture).
//
// What it replaces, for a whole batch of frames resident in HBM:
//   LaneDetector.draw_lanes                      /root/reference/src/perception/lane_detector.py:220-251
//       cv2.fillPoly on a copy + cv2.addWeighted(frame, 0.7, overlay, 0.3, 0) + cv2.polylines(.., thickness 3)
//   OverlayRenderer.draw_lane_offset_indicator   /root/reference/src/visualization/overlays.py:103-148
//       cv2.rectangle (filled, outlined), cv2.line, filled cv2.circle, cv2.putText (as a host-rendered bit mask)
//   SyntheticDataGenerator.generate_frame_with_vehicles (bytecode only, SURVEY Appendix B)
//       cv2.line (thickness 1 and 2), cv2.rectangle, cv2.fillPoly, filled cv2.circle
//
// Two layers.  The host layer (draw_prims.h, plain C++) turns cv2-level calls into row-separable device primitives with
// OpenCV 4.13's own integer / double arithmetic (clipLine's truncating double division, Bresenham end points, the
// 16.16 DDA that outlines FillConvexPoly, FillConvexPoly's rounded edge steps, the pre-clip of thick segments against the
// image grown by `thickness`, ThickLine's cvRound'ed normal, the midpoint circle, fillPoly's edge table built from the
// clipped end points) -- restated in oracle/draw.py and pinned there against cv2 itself.  The device layer rasterises:
// one CTA per (band of rows, frame) walks the frame's primitive list in order (painter's order is what cv2 gives), a
// barrier between primitives that touch the band; inside a primitive every row / point is independent:
//   TRAP      rows y0..y1 of a trapezoid with 16.16 edges  -> 16-byte stores of the 3-byte colour pattern
//   ROWS      consecutive full-width rows, one colour each (the generator's sky gradient: 540 cv2.line calls)
//   LINE8     8-connected Bresenham line, point i in closed form: minor = (2*dmin*i + dmaj - 1) / (2*dmaj)
//   LINE2     16.16 DDA line, point i in closed form
//   POLYFILL  fillPoly's scan conversion: a warp per row gathers the active edges, orders their x, fills the pairs
//   MASK_BEGIN .. MASK_BLEND   the primitives in between set bits of a shared-memory coverage mask of the band instead
//             of writing pixels; MASK_BLEND then applies cv2.addWeighted's float32 fma(a, alpha, fma(b, beta, gamma))
//             once per covered pixel (a pixel on the polygon outline AND inside it is blended once, as cv2's overlay is)
//   BITMAP    1-bit mask blit (text)
// The lane overlay has its own kernel (k7_lanes, below) that needs no primitive lists: the geometry core of draw_prims.h
// is host/device code, and a thread runs it for one polygon edge or thick segment and rasterises directly.
// Entry points: lane_draw_commands, lane_draw_lanes_batch, lane_draw_lanes_records, lane_generate_frames.
// HBM-bound byte work: no tensor cores, no GEMM shapes.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <thread>
#include <vector>

#include "draw_prims.h"
#include "host_stage.h"

using namespace lane_draw;

namespace {

// ------------------------------------------------------------------------------------------------ device side
struct Target {
    uint8_t *frame;      // this frame
    uint32_t *mask;      // band mask in shared memory
    int H, W, WW;        // WW = words per mask row
    int by0, by1;        // band rows [by0, by1]
    bool to_mask;
};

__device__ __forceinline__ uint32_t pattern_word(uint32_t color, int q)   // 4 bytes of the BGR pattern starting at channel q
{
    const uint32_t c0 = color & 255, c1 = (color >> 8) & 255, c2 = (color >> 16) & 255;
    const uint32_t w0 = c0 | c1 << 8 | c2 << 16 | c0 << 24, w1 = c1 | c2 << 8 | c0 << 16 | c1 << 24,
                   w2 = c2 | c0 << 8 | c1 << 16 | c2 << 24;
    return q == 0 ? w0 : q == 1 ? w1 : w2;
}

// pixels x1..x2 (already clipped, x1 <= x2) of row y, by one warp
__device__ void warp_span(const Target &t, int y, int x1, int x2, uint32_t color, int lane)
{
    if (t.to_mask) {
        uint32_t *row = t.mask + (size_t)(y - t.by0) * t.WW;
        const int w1 = x1 >> 5, w2 = x2 >> 5;
        for (int w = w1 + lane; w <= w2; w += 32) {
            uint32_t m = 0xffffffffu;
            if (w == w1) m &= 0xffffffffu << (x1 & 31);
            if (w == w2) m &= 0xffffffffu >> (31 - (x2 & 31));
            atomicOr(row + w, m);
        }
        return;
    }
    uint8_t *row = t.frame + (size_t)y * t.W * 3;
    const long b0 = 3L * x1, b1 = 3L * x2 + 3;
    const uintptr_t base = (uintptr_t)row;
    long al = (long)(((base + b0 + 15) & ~(uintptr_t)15) - base);
    if (al > b1) al = b1;
    if (lane < al - b0) {
        const long o = b0 + lane;
        row[o] = (uint8_t)(color >> (8 * (o % 3)));
    }
    const long nvec = (b1 - al) >> 4;
    for (long v = lane; v < nvec; v += 32) {
        const long o = al + 16 * v;
        const int q = (int)(o % 3);
        uint4 val;
        val.x = pattern_word(color, q);
        val.y = pattern_word(color, (q + 1) % 3);
        val.z = pattern_word(color, (q + 2) % 3);
        val.w = val.x;
        *(uint4 *)(row + o) = val;
    }
    const long t0 = al + 16 * nvec;
    if (lane < b1 - t0) {
        const long o = t0 + lane;
        row[o] = (uint8_t)(color >> (8 * (o % 3)));
    }
}

__device__ __forceinline__ void plot(const Target &t, int x, int y, uint32_t color)
{
    if ((unsigned)x >= (unsigned)t.W || y < t.by0 || y > t.by1) return;
    if (t.to_mask) {
        atomicOr(t.mask + (size_t)(y - t.by0) * t.WW + (x >> 5), 1u << (x & 31));
    } else {
        uint8_t *p = t.frame + ((size_t)y * t.W + x) * 3;
        p[0] = (uint8_t)color;
        p[1] = (uint8_t)(color >> 8);
        p[2] = (uint8_t)(color >> 16);
    }
}

__device__ __forceinline__ void clipped_span(const Target &t, int y, long x1, long x2, uint32_t color, int lane)
{
    if (x2 >= 0 && x1 < t.W) {
        if (x1 < 0) x1 = 0;
        if (x2 >= t.W) x2 = t.W - 1;
        if (x1 <= x2) warp_span(t, y, (int)x1, (int)x2, color, lane);
    }
}

// fillPoly's scan conversion of rows ya..yb: a warp per row gathers the active edges (y0 <= y < y1), orders their
// x = x0 + (y - y0) * dx and fills [ceil(x_a), floor(x_b)] for every pair.  edges: (y0, y1, x, dx) per edge.
__device__ void polyfill_rows(const Target &t, const int64_t *edges, int ne, int ya, int yb, uint32_t color, int warp, int nwarps,
                              int lane, int64_t *row_x)
{
    for (int y = ya + warp; y <= yb; y += nwarps) {
        int n = 0;
        for (int e0 = 0; e0 < ne; e0 += 32) {
            const int e = e0 + lane;
            bool act = false;
            int64_t x = 0;
            if (e < ne) {
                const int64_t ey0 = edges[4 * e], ey1 = edges[4 * e + 1];
                act = ey0 <= y && y < ey1;
                if (act) x = edges[4 * e + 2] + (y - ey0) * edges[4 * e + 3];
            }
            const unsigned m = __ballot_sync(0xffffffffu, act);
            const int pos = n + __popc(m & ((1u << lane) - 1));
            if (act && pos < MAX_ROW_EDGES) row_x[pos] = x;
            n += __popc(m);
        }
        n = min(n, MAX_ROW_EDGES);
        __syncwarp();
        // rank sort (n is 2 for a simple polygon)
        int64_t mine[MAX_ROW_EDGES / 32];
        int rank[MAX_ROW_EDGES / 32];
#pragma unroll
        for (int j = 0; j < MAX_ROW_EDGES / 32; j++) {
            const int i = lane + 32 * j;
            rank[j] = 0;
            if (i < n) {
                mine[j] = row_x[i];
                for (int k = 0; k < n; k++) {
                    const int64_t o = row_x[k];
                    rank[j] += (o < mine[j]) || (o == mine[j] && k < i);
                }
            }
        }
        __syncwarp();
#pragma unroll
        for (int j = 0; j < MAX_ROW_EDGES / 32; j++)
            if (lane + 32 * j < n) row_x[rank[j]] = mine[j];
        __syncwarp();
        for (int k = 0; k + 1 < n; k += 2)
            clipped_span(t, y, (long)((row_x[k] + XY_ONE - 1) >> XY_SHIFT), (long)(row_x[k + 1] >> XY_SHIFT), color, lane);
        __syncwarp();
    }
}

// cv2.addWeighted(img, alpha, overlay, beta, gamma) on rows ya..yb, columns x0..x1: overlay = color where the band mask is set
__device__ void mask_blend(const Target &t, int ya, int yb, int x0, int x1, uint32_t color, float alpha, float beta, float gamma,
                           bool outside_too, int tid)
{
    const int bw = x1 - x0 + 1, total = (yb - ya + 1) * bw;
    for (int i = tid; i < total; i += DRAW_THREADS) {
        const int y = ya + i / bw, x = x0 + i % bw;
        const bool in = (t.mask[(size_t)(y - t.by0) * t.WW + (x >> 5)] >> (x & 31)) & 1;
        if (!in && !outside_too) continue;
        uint8_t *px = t.frame + ((size_t)y * t.W + x) * 3;
#pragma unroll
        for (int ch = 0; ch < 3; ch++) {
            const float a = (float)px[ch];
            const float o = in ? (float)((color >> (8 * ch)) & 255) : a;
            const int r = __float2int_rn(fmaf(a, alpha, fmaf(o, beta, gamma)));
            px[ch] = (uint8_t)min(255, max(0, r));
        }
    }
}

__global__ void __launch_bounds__(DRAW_THREADS) k7_draw(uint8_t *frames, const Prim *prims, const int64_t *band_begin,
                                                       const int32_t *band_idx, const int64_t *side, int H, int W)
{
    extern __shared__ uint32_t smem[];
    const int f = blockIdx.y, band = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = DRAW_THREADS / 32;
    Target t;
    t.frame = frames + (size_t)f * H * W * 3;
    t.H = H; t.W = W; t.WW = (W + 31) >> 5;
    t.by0 = band * BAND_ROWS;
    t.by1 = min(H, t.by0 + BAND_ROWS) - 1;
    t.mask = smem;
    t.to_mask = false;
    int64_t *row_x = (int64_t *)(smem + (size_t)BAND_ROWS * t.WW + (((size_t)BAND_ROWS * t.WW) & 1)) + warp * MAX_ROW_EDGES;

    // the primitives of this frame that touch this band, in drawing order (binned on the host)
    const int64_t p_end = band_begin[(size_t)f * gridDim.x + band + 1];
    // Painter's order only matters between primitives that may write DIFFERENT values to one pixel: a run of primitives of
    // one colour (the ~14 pieces of a thick segment, a polygon's outline and interior) commutes, and so does anything that
    // only sets mask bits.  `pending` = colour drawn since the last barrier (NO_COLOUR: nothing, MIXED: per-row colours).
    constexpr uint32_t NO_COLOUR = 0xFFFFFFFFu, MIXED = 0xFFFFFFFEu;
    uint32_t pending = NO_COLOUR;
    for (int64_t pi = band_begin[(size_t)f * gridDim.x + band]; pi < p_end; pi++) {
        const Prim p = prims[band_idx[pi]];
        if (p.op == P_MASK_BEGIN) {              // band-uniform state: no row test
            pending = NO_COLOUR;
            __syncthreads();
            for (int i = tid; i < BAND_ROWS * t.WW; i += DRAW_THREADS) t.mask[i] = 0;
            t.to_mask = true;
            __syncthreads();
            continue;
        }
        const int ya = max(p.y0, t.by0), yb = min(p.y1, t.by1);
        if (p.op == P_MASK_BLEND) {
            pending = NO_COLOUR;
            __syncthreads();
            t.to_mask = false;
            if (ya <= yb)
                mask_blend(t, ya, yb, (int)p.c, (int)p.d, p.color, __int_as_float((int)(uint32_t)p.a),
                           __int_as_float((int)(uint32_t)(p.a >> 32)), __int_as_float((int)(uint32_t)p.b), (p.b >> 32) & 1, tid);
            __syncthreads();
            continue;
        }
        if (ya > yb) continue;
        if (!t.to_mask) {
            const uint32_t mine = p.op == P_ROWS ? MIXED : p.color;
            if (pending != NO_COLOUR && (pending != mine || mine == MIXED)) __syncthreads();
            pending = mine;
        }
        switch (p.op) {
        case P_TRAP:
            for (int y = ya + warp; y <= yb; y += nwarps) {
                int64_t l = p.a + (int64_t)(y - p.y0) * p.b, r = p.c + (int64_t)(y - p.y0) * p.d;
                if (l > r) { const int64_t s = l; l = r; r = s; }
                clipped_span(t, y, (long)((l + HALF) >> XY_SHIFT), (long)((r + HALF) >> XY_SHIFT), p.color, lane);
            }
            break;
        case P_ROWS: {
            const uint32_t *colors = (const uint32_t *)(side + p.a);
            const int x1 = (int)p.b, x2 = (int)p.c;
            for (int y = ya + warp; y <= yb; y += nwarps) clipped_span(t, y, x1, x2, colors[y - p.y0 + (int)p.d], lane);
            break;
        }
        case P_LINE8: {
            const int x1 = (int)(p.a >> 32), y1 = (int)(uint32_t)p.a;
            const int dmaj = (int)(p.b >> 32), dmin = (int)(uint32_t)p.b;
            const bool vert = p.c & 1;
            const int sy = (p.c & 2) ? -1 : 1;
            for (int i = tid; i <= dmaj; i += DRAW_THREADS) {
                const int k = dmaj ? (int)((2LL * dmin * i + dmaj - 1) / (2LL * dmaj)) : 0;
                if (vert) plot(t, x1 + k, y1 + sy * i, p.color);
                else plot(t, x1 + i, y1 + sy * k, p.color);
            }
            break;
        }
        case P_LINE2: {
            const int m0 = (int)(p.a >> 32), count = (int)(uint32_t)p.a;
            for (int i = tid; i < count; i += DRAW_THREADS) {
                const int minor = (int)((p.b + (int64_t)i * p.c) >> XY_SHIFT);
                if (p.d & 1) plot(t, m0 + i, minor, p.color);
                else plot(t, minor, m0 + i, p.color);
            }
            break;
        }
        case P_POLYFILL:
            polyfill_rows(t, side + p.a, (int)p.b, ya, yb, p.color, warp, nwarps, lane, row_x);
            break;
        case P_BITMAP: {
            const uint32_t *bits = (const uint32_t *)(side + p.a);
            const int bx = (int)(p.b >> 32), by = (int)(uint32_t)p.b, bw = (int)(p.c >> 32), bh = (int)(uint32_t)p.c;
            const int wpr = (bw + 31) >> 5;
            (void)bh;
            for (int i = tid; i < (yb - ya + 1) * wpr; i += DRAW_THREADS) {
                const int y = ya + i / wpr, w = i % wpr;
                uint32_t m = bits[(size_t)(y - by) * wpr + w];
                while (m) {
                    const int b = __ffs(m) - 1;
                    m &= m - 1;
                    plot(t, bx + 32 * w + b, y, p.color);
                }
            }
            break;
        }
        default: break;
        }
    }
}

// ---- k7_lanes: LaneDetector.draw_lanes for a batch without any host expansion ------------------------------------------
// The overlay of one frame is 100 polygon edges and 98 thick segments.  A CTA (band of rows, frame) reads the frame's two
// 50-point polylines (from the lane records on the device, or from an uploaded copy of LaneLine.points), and every thread
// runs OpenCV's arithmetic for ONE edge / segment with the geometry core of draw_prims.h -- the same template functions
// the host half expands primitives with -- and rasterises what falls into its band directly:
//   1. polygon outline (Line per edge) and scan conversion (edge table in shared memory, a warp per row) into the band's
//      coverage mask, then one addWeighted blend per covered pixel;
//   2. the left polyline's segments (quadrilateral by FillConvexPoly's row runs, its DDA outline, the end caps), all one
//      colour, so no ordering between threads; 3. a barrier, then the right polyline's.
// Three barriers per band instead of one per primitive, and 800 bytes per frame instead of 75 KB of primitive lists.
struct LaneSrc {                     // where the points / validity flags of frame f, side s live
    const char *base;
    size_t frame_stride, pts_off[2], valid_off[2];
    int valid_bytes;                 // 1: uint8 flags, 4: int32 (lane_side.valid)
};

struct DevEmit {                     // emitter of the geometry core: rasterise into this CTA's band (or its mask)
    Target t;
    uint32_t color;
    int W, H;
    __device__ void span(int64_t y, int64_t x1, int64_t x2)
    {
        if (y < t.by0 || y > t.by1 || x2 < 0 || x1 >= W || x1 > x2) return;
        if (x1 < 0) x1 = 0;
        if (x2 >= W) x2 = W - 1;
        for (int64_t x = x1; x <= x2; x++) plot(t, (int)x, (int)y, color);
    }
    __device__ void line8(int64_t x1, int64_t y1, int64_t dmaj, int64_t dmin, bool vert, int sy)
    {
        for (int64_t i = 0; i <= dmaj; i++) {
            const int64_t k = dmaj ? (2 * dmin * i + dmaj - 1) / (2 * dmaj) : 0;
            if (vert) plot(t, (int)(x1 + k), (int)(y1 + sy * i), color);
            else plot(t, (int)(x1 + i), (int)(y1 + sy * k), color);
        }
    }
    __device__ void line2(bool xmajor, int64_t major0, int64_t count, int64_t minor0, int64_t step)
    {
        for (int64_t i = 0; i < count; i++) {
            const int64_t minor = (minor0 + i * step) >> XY_SHIFT;
            if (minor < 0 || minor >= 32768) continue;          // outside any supported frame
            if (xmajor) plot(t, (int)(major0 + i), (int)minor, color);
            else plot(t, (int)minor, (int)(major0 + i), color);
        }
    }
    __device__ void trap(int64_t y0, int64_t y1, int64_t xl0, int64_t dxl, int64_t xr0, int64_t dxr)
    {
        const int64_t ya = y0 > t.by0 ? y0 : t.by0, yb = y1 < t.by1 ? y1 : t.by1;
        for (int64_t y = ya; y <= yb; y++) {
            int64_t l = xl0 + (y - y0) * dxl, r = xr0 + (y - y0) * dxr;
            if (l > r) { const int64_t s = l; l = r; r = s; }
            span(y, (l + HALF) >> XY_SHIFT, (r + HALF) >> XY_SHIFT);
        }
    }
};

constexpr int LANE_PTS = 50;

__global__ void __launch_bounds__(DRAW_THREADS) k7_lanes(uint8_t *frames, LaneSrc src, int H, int W, int fill_lane, uint32_t fill_color,
                                                        uint32_t left_color, uint32_t right_color, float alpha, float beta)
{
    extern __shared__ uint32_t smem[];
    __shared__ int32_t s_pts[2][LANE_PTS][2];
    __shared__ int s_valid[2];
    __shared__ __align__(8) int64_t s_edges[2 * LANE_PTS][4];
    __shared__ int s_fill[7];        // blend here?, its rows ya..yb and columns x0..x1, scan-conversion rows
    const int f = blockIdx.y, band = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = DRAW_THREADS / 32;
    Target t;
    t.frame = frames + (size_t)f * H * W * 3;
    t.H = H; t.W = W; t.WW = (W + 31) >> 5;
    t.by0 = band * BAND_ROWS;
    t.by1 = min(H, t.by0 + BAND_ROWS) - 1;
    t.mask = smem;
    t.to_mask = false;
    int64_t *row_x = (int64_t *)(smem + (size_t)BAND_ROWS * t.WW + (((size_t)BAND_ROWS * t.WW) & 1)) + warp * MAX_ROW_EDGES;
    const char *rec = src.base + (size_t)f * src.frame_stride;
    if (tid < 2) s_valid[tid] = src.valid_bytes == 1 ? (int)*(const uint8_t *)(rec + src.valid_off[tid]) : *(const int32_t *)(rec + src.valid_off[tid]);
    for (int i = tid; i < 2 * LANE_PTS * 2; i += DRAW_THREADS) {
        const int s = i / (LANE_PTS * 2), k = i - s * LANE_PTS * 2;
        (&s_pts[s][0][0])[k] = ((const int32_t *)(rec + src.pts_off[s]))[k];
    }
    __syncthreads();
    const bool lv = s_valid[0] != 0, rv = s_valid[1] != 0;
    auto vertex = [&](int i) {       // pts = vstack([left.points, right.points[::-1]])   lane_detector.py:242
        return i < LANE_PTS ? Pt{s_pts[0][i][0], s_pts[0][i][1]} : Pt{s_pts[1][2 * LANE_PTS - 1 - i][0], s_pts[1][2 * LANE_PTS - 1 - i][1]};
    };
    if (fill_lane && lv && rv) {
        // the polygon's bounding box decides whether this band has anything to blend (the blend leaves other pixels alone)
        if (tid == 0) {
            int64_t y0 = INT64_MAX, y1 = INT64_MIN, x0 = INT64_MAX, x1 = INT64_MIN;
            for (int i = 0; i < 2 * LANE_PTS; i++) {
                const Pt v = vertex(i);
                y0 = lane_min(y0, v.y); y1 = lane_max(y1, v.y); x0 = lane_min(x0, v.x); x1 = lane_max(x1, v.x);
            }
            y0 = lane_max<int64_t>(y0, t.by0); y1 = lane_min<int64_t>(y1, t.by1);
            x0 = lane_max<int64_t>(x0, 0); x1 = lane_min<int64_t>(x1, W - 1);
            s_fill[0] = y0 <= y1 && x0 <= x1;
            s_fill[1] = (int)y0; s_fill[2] = (int)y1; s_fill[3] = (int)x0; s_fill[4] = (int)x1;
        }
        __syncthreads();
        if (s_fill[0]) {
            for (int i = tid; i < BAND_ROWS * t.WW; i += DRAW_THREADS) t.mask[i] = 0;
            __syncthreads();
            t.to_mask = true;
            if (tid < 2 * LANE_PTS) {            // CollectPolyEdges: the outline into the mask, the edge record into shared memory
                Pt t0, t1;
                PolyEdge e;
                const bool has = geo_poly_edge(W, H, vertex(tid ? tid - 1 : 2 * LANE_PTS - 1), vertex(tid), t0, t1, e);
                DevEmit em{t, fill_color, W, H};
                geo_line8(em, t0, t1);
                s_edges[tid][0] = has ? e.y0 : 0; s_edges[tid][1] = has ? e.y1 : 0;      // y0 == y1: never active
                s_edges[tid][2] = e.x; s_edges[tid][3] = e.dx;
                if (!has) { s_edges[tid][2] = 0; s_edges[tid][3] = 0; }
            }
            __syncthreads();
            if (tid == 0) {                      // FillEdgeCollection's early-outs and row range
                int total = 0;
                int64_t y_min = INT64_MAX, y_max = INT64_MIN, x_min = INT64_MAX, x_max = INT64_MIN;
                for (int i = 0; i < 2 * LANE_PTS; i++) {
                    if (s_edges[i][0] == s_edges[i][1]) continue;
                    total++;
                    const int64_t xe = s_edges[i][2] + (s_edges[i][1] - s_edges[i][0]) * s_edges[i][3];
                    y_min = lane_min(y_min, s_edges[i][0]); y_max = lane_max(y_max, s_edges[i][1]);
                    x_min = lane_min(x_min, lane_min(s_edges[i][2], xe)); x_max = lane_max(x_max, lane_max(s_edges[i][2], xe));
                }
                bool run = total >= 2 && !(y_max < 0 || y_min >= H || x_max < 0 || x_min >= ((int64_t)W << XY_SHIFT));
                const int64_t ya = lane_max<int64_t>(lane_max<int64_t>(y_min, 0), t.by0), yb = lane_min<int64_t>(lane_min<int64_t>(y_max, H) - 1, t.by1);
                s_fill[0] = run && ya <= yb ? 1 : 2;                 // 2: outline only
                s_fill[5] = (int)ya; s_fill[6] = (int)yb;
            }
            __syncthreads();
            if (s_fill[0] == 1)
                polyfill_rows(t, &s_edges[0][0], 2 * LANE_PTS, s_fill[5], s_fill[6], fill_color, warp, nwarps, lane, row_x);
            __syncthreads();
            t.to_mask = false;
            mask_blend(t, s_fill[1], s_fill[2], s_fill[3], s_fill[4], fill_color, alpha, beta, 0.0f, false, tid);
        }
        __syncthreads();
    }
    // cv2.polylines(frame, [points], False, colour, 3): segment s is ThickLine(p[s], p[s+1], 3, flags = 3 for the first, else 2)
    for (int side = 0; side < 2; side++) {
        if (side == 0 ? lv : rv) {
            if (tid < LANE_PTS - 1) {
                const Pt p0{s_pts[side][tid][0], s_pts[side][tid][1]}, p1{s_pts[side][tid + 1][0], s_pts[side][tid + 1][1]};
                const int64_t lo = lane_min(p0.y, p1.y) - 4, hi = lane_max(p0.y, p1.y) + 4;      // half width 2 + cap radius 1
                if (hi >= t.by0 && lo <= t.by1) {
                    DevEmit em{t, side == 0 ? left_color : right_color, W, H};
                    geo_thick_line(em, p0, p1, 3, tid == 0 ? 3 : 2);
                }
            }
        }
        __syncthreads();
    }
}

struct Chunk {
    Builder b;
    int f0 = 0, f1 = 0;
    const char *err = nullptr;
    std::vector<int32_t> counts;      // [frames of the chunk][bands]: primitives that touch the band
    int64_t prim_base = 0, side_base = 0;
};

inline int band_lo(const Prim &p) { return p.y0 / BAND_ROWS; }
inline int band_hi(const Prim &p) { return p.y1 / BAND_ROWS; }

// launch(d_frames, d_frames) on frames that are drawn on in place: device frames directly, host frames through the
// device's scratch (cleared there instead of uploaded when `clear_first`).  Blocking either way.
template <class Launch>
int draw_frames(const char *who, uint8_t *frames, int on_device, size_t bytes, int device, cudaStream_t st, bool clear_first,
                Launch &&launch)
{
    if (!on_device) return lane_host_round_trip(who, device, st, clear_first ? nullptr : frames, bytes, frames, bytes, launch);
    const int rc = launch(frames, frames);
    const cudaError_t e = cudaStreamSynchronize(st);
    return rc ? rc : e ? lane_api_fail(LANE_ERR_CUDA, who, "synchronise", e) : LANE_OK;
}

// The host half, frames in parallel: worker t expands the drawing calls of its frames into primitives and counts them per
// band; the lists are then laid out in one pinned block (band offsets | primitives | side tables | per-band index lists),
// filled by the same workers, and uploaded with one copy.  build_frame(Builder&, int f, const char **err) -> bool.
template <class BuildFrame>
int draw_driver(const char *who, uint8_t *frames, int on_device, int n, int H, int W, int device, cudaStream_t st,
                float *device_ms, BuildFrame build_frame, bool clear_first = false)
{
    const int bands = (H + BAND_ROWS - 1) / BAND_ROWS;
    const int T = std::max(1, std::min({n / 8, (int)std::thread::hardware_concurrency(), 16}));
    std::vector<Chunk> chunks(T);
    auto for_chunks = [&](auto fn) {
        std::vector<std::thread> th;
        for (int t = 1; t < T; t++) th.emplace_back([&, t] { fn(chunks[t]); });
        fn(chunks[0]);
        for (auto &x : th) x.join();
    };
    for (int t = 0; t < T; t++) {
        chunks[t].f0 = (int)((int64_t)n * t / T);
        chunks[t].f1 = (int)((int64_t)n * (t + 1) / T);
        chunks[t].b.H = H;
        chunks[t].b.W = W;
    }
    for_chunks([&](Chunk &c) {
        c.counts.assign((size_t)(c.f1 - c.f0) * bands, 0);
        for (int f = c.f0; f < c.f1; f++) {
            c.b.begin.push_back((int64_t)c.b.prims.size());
            if (!build_frame(c.b, f, &c.err)) return;
            int32_t *cnt = c.counts.data() + (size_t)(f - c.f0) * bands;
            for (size_t i = (size_t)c.b.begin.back(); i < c.b.prims.size(); i++)
                for (int bd = band_lo(c.b.prims[i]); bd <= band_hi(c.b.prims[i]); bd++) cnt[bd]++;
        }
        c.b.begin.push_back((int64_t)c.b.prims.size());
    });
    for (const Chunk &c : chunks)
        if (c.err) return lane_api_fail(LANE_ERR_INVALID, who, c.err);
    int64_t n_prims = 0, n_side = 0;
    for (Chunk &c : chunks) {
        c.prim_base = n_prims;
        c.side_base = n_side;
        n_prims += (int64_t)c.b.prims.size();
        n_side += (int64_t)((c.b.side.size() + 1) & ~(size_t)1);
    }
    std::vector<int64_t> band_begin((size_t)n * bands + 1);
    int64_t n_idx = 0;
    for (const Chunk &c : chunks)
        for (size_t k = 0; k < c.counts.size(); k++) {
            band_begin[(size_t)c.f0 * bands + k] = n_idx;
            n_idx += c.counts[k];
        }
    band_begin[(size_t)n * bands] = n_idx;
    const size_t nb_begin = band_begin.size() * 8, nb_prims = (size_t)n_prims * sizeof(Prim), nb_side = (size_t)std::max<int64_t>(n_side, 1) * 8,
                 nb_idx = (size_t)std::max<int64_t>(n_idx, 1) * 4;
    const size_t off_prims = (nb_begin + 63) & ~(size_t)63, off_side = (off_prims + nb_prims + 63) & ~(size_t)63,
                 off_idx = (off_side + nb_side + 63) & ~(size_t)63, total = off_idx + nb_idx;

    LaneDeviceHost &dh = lane_device_host(device);
    std::lock_guard<std::mutex> lk(dh.draw_mu);
    // write-combined: the block is written once, front to back, by up to 16 host threads and then read by the copy
    // engine only.  (Measured on the B200 box: the upload that follows the fill runs at ~11 GB/s with write-combined
    // and with ordinary pinned memory alike, a repeated upload of the same block at 46 GB/s -- the hand-over from the
    // CPU's writes to the DMA reads is what costs, 2 ms per 22 MB; LANE_B200_DRAW_DEBUG=1 prints it.)
    if (dh.reserve_draw(total, std::max(total + total / 2, (size_t)1 << 20)))
        return lane_api_fail(LANE_ERR_CUDA, who, "staging allocation failed");
    uint8_t *h = dh.draw_h, *d = dh.draw_d;
    memcpy(h, band_begin.data(), nb_begin);
    for_chunks([&](Chunk &ck) {
        Prim *hp = (Prim *)(h + off_prims) + ck.prim_base;
        int64_t *hs = (int64_t *)(h + off_side) + ck.side_base;
        int32_t *hi = (int32_t *)(h + off_idx);
        if (!ck.b.side.empty()) memcpy(hs, ck.b.side.data(), ck.b.side.size() * 8);
        // the chunk's index lists are one contiguous stretch of the block: filled in ordinary memory (scattered 4-byte
        // writes), then copied out in one sweep
        const int64_t idx0 = band_begin[(size_t)ck.f0 * bands], idx1 = band_begin[(size_t)ck.f1 * bands];
        std::vector<int32_t> local((size_t)(idx1 - idx0));
        std::vector<int64_t> cursor(bands);
        for (int f = ck.f0; f < ck.f1; f++) {
            for (int bd = 0; bd < bands; bd++) cursor[bd] = band_begin[(size_t)f * bands + bd] - idx0;
            for (int64_t i = ck.b.begin[f - ck.f0]; i < ck.b.begin[f - ck.f0 + 1]; i++) {
                Prim p = ck.b.prims[i];
                if (p.op == P_ROWS || p.op == P_POLYFILL || p.op == P_BITMAP) p.a += ck.side_base;
                hp[i] = p;
                for (int bd = band_lo(p); bd <= band_hi(p); bd++) local[cursor[bd]++] = (int32_t)(ck.prim_base + i);
            }
        }
        if (!local.empty()) memcpy(hi + idx0, local.data(), local.size() * 4);
    });

    CudaEvent e0, e1, ec;
    static const bool dbg = getenv("LANE_B200_DRAW_DEBUG") != nullptr;
    auto launch = [&](uint8_t *d_frames, uint8_t *) {
        if (device_ms) { e0.create(); e1.create(); cudaEventRecord(e0, st); }
        if (clear_first) cudaMemsetAsync(d_frames, 0, (size_t)n * H * W * 3, st);
        cudaMemcpyAsync(d, h, total, cudaMemcpyHostToDevice, st);
        if (dbg && device_ms) { ec.create(); cudaEventRecord(ec, st); }
        const int WW = (W + 31) >> 5;
        const size_t mask_words = (size_t)BAND_ROWS * WW;
        const size_t smem = (mask_words + (mask_words & 1)) * 4 + (size_t)(DRAW_THREADS / 32) * MAX_ROW_EDGES * 8;
        static bool configured[LANE_MAX_DEVICES];
        if (smem > 48 * 1024 && !configured[device]) {
            cudaFuncSetAttribute(k7_draw, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
            configured[device] = true;
        }
        if (smem > 200 * 1024) return lane_api_fail(LANE_ERR_UNSUPPORTED, who, "frame too wide for the band mask");
        k7_draw<<<dim3(bands, n), DRAW_THREADS, smem, st>>>(d_frames, (const Prim *)(d + off_prims), (const int64_t *)d,
                                                            (const int32_t *)(d + off_idx), (const int64_t *)(d + off_side), H, W);
        const cudaError_t e = cudaGetLastError();
        if (device_ms) cudaEventRecord(e1, st);
        return e ? lane_api_fail(LANE_ERR_CUDA, who, "k7_draw launch", e) : LANE_OK;
    };
    int rc = draw_frames(who, frames, on_device, (size_t)n * H * W * 3, device, st, clear_first, launch);
    if (rc == LANE_OK && device_ms) cudaEventElapsedTime(device_ms, e0, e1);
    if (ec) {
        float cms = 0;
        if (rc == LANE_OK) cudaEventElapsedTime(&cms, e0, ec);
        fprintf(stderr, "lane_draw: %lld primitives, %lld band entries, %.2f MB uploaded in %.3f ms, upload + kernel %.3f ms, %d host threads\n",
                (long long)n_prims, (long long)n_idx, total / 1e6, cms, device_ms ? *device_ms : 0.f, T);
    }
    return rc;
}

}  // namespace

extern "C" int lane_draw_commands(uint8_t *frames, int on_device, int n, int height, int width, const int32_t *commands,
                                  const int64_t *command_begin, int device, void *cuda_stream, float *device_ms)
{
    constexpr const char *who = "lane_draw_commands";
    if (!frames || !commands || !command_begin || n < 1 || height < 1 || width < 1)
        return lane_api_fail(LANE_ERR_INVALID, who, "bad arguments");
    if (height > 32767 || width > 32767) return lane_api_fail(LANE_ERR_UNSUPPORTED, who, "frame larger than 32767 px");
    for (int f = 0; f < n; f++)
        if (command_begin[f + 1] < command_begin[f]) return lane_api_fail(LANE_ERR_INVALID, who, "command_begin must not decrease");
    if (int rc = lane_api_device(who, device)) return rc;
    return draw_driver(who, frames, on_device, n, height, width, device, (cudaStream_t)cuda_stream, device_ms,
                       [&](Builder &b, int f, const char **err) {
                           return parse_commands(b, commands + command_begin[f], command_begin[f + 1] - command_begin[f], err);
                       });
}

namespace {

struct LaneItem {                    // what k7_lanes reads per frame when the lanes come from the host
    int32_t pts[2][LANE_PTS][2];
    int32_t valid[2];
};

int launch_lanes(const char *who, uint8_t *d_frames, const LaneSrc &src, int n, int H, int W, int fill_lane, cudaStream_t st,
                 int device)
{
    const int bands = (H + BAND_ROWS - 1) / BAND_ROWS, WW = (W + 31) >> 5;
    const size_t mask_words = (size_t)BAND_ROWS * WW;
    const size_t smem = (mask_words + (mask_words & 1)) * 4 + (size_t)(DRAW_THREADS / 32) * MAX_ROW_EDGES * 8;
    static bool configured[LANE_MAX_DEVICES];
    if (smem > 44 * 1024 && !configured[device]) {
        cudaFuncSetAttribute(k7_lanes, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        configured[device] = true;
    }
    if (smem > 200 * 1024) return lane_api_fail(LANE_ERR_UNSUPPORTED, who, "frame too wide for the band mask");
    // (0, 255, 100) at weight 0.3 over 0.7 (lane_detector.py:243-244), left (255, 0, 0) :248, right (0, 0, 255) :251
    k7_lanes<<<dim3(bands, n), DRAW_THREADS, smem, st>>>(d_frames, src, H, W, fill_lane, 0u | 255u << 8 | 100u << 16, 255u, 255u << 16,
                                                        0.7f, 0.3f);
    const cudaError_t e = cudaGetLastError();
    return e ? lane_api_fail(LANE_ERR_CUDA, who, "k7_lanes launch", e) : LANE_OK;
}

bool lanes_by_primitives()           // LANE_B200_DRAW_LANES=prims: the host-expanded primitive lists (A/B, and the tests run both)
{
    const char *e = getenv("LANE_B200_DRAW_LANES");
    return e && !strcmp(e, "prims");
}

}  // namespace

extern "C" int lane_draw_lanes_batch(uint8_t *frames, int on_device, int n, int height, int width, const int32_t *left_points,
                                     const uint8_t *left_valid, const int32_t *right_points, const uint8_t *right_valid,
                                     int fill_lane, int device, void *cuda_stream, float *device_ms)
{
    constexpr const char *who = "lane_draw_lanes_batch";
    if (!frames || !left_points || !right_points || !left_valid || !right_valid || n < 1 || height < 1 || width < 1)
        return lane_api_fail(LANE_ERR_INVALID, who, "bad arguments");
    if (height > 32767 || width > 32767) return lane_api_fail(LANE_ERR_UNSUPPORTED, who, "frame larger than 32767 px");
    if (int rc = lane_api_device(who, device)) return rc;
    cudaStream_t st = (cudaStream_t)cuda_stream;
    if (lanes_by_primitives())
        return draw_driver(who, frames, on_device, n, height, width, device, st, device_ms,
                           [&](Builder &b, int f, const char **) {
                               build_draw_lanes_frame(b, left_points + (size_t)f * LANE_NUM_POINTS * 2, left_valid[f],
                                                      right_points + (size_t)f * LANE_NUM_POINTS * 2, right_valid[f], fill_lane);
                               return true;
                           });
    // default: the geometry runs on the device (k7_lanes); only the 100 points per frame are uploaded
    const size_t item_bytes = (size_t)n * sizeof(LaneItem);
    LaneDeviceHost &dh = lane_device_host(device);
    std::lock_guard<std::mutex> lk(dh.draw_mu);
    if (dh.reserve_draw(item_bytes, std::max(item_bytes * 2, (size_t)1 << 20)))
        return lane_api_fail(LANE_ERR_CUDA, who, "staging allocation failed");
    uint8_t *h = dh.draw_h, *d = dh.draw_d;
    LaneItem *items = (LaneItem *)h;
    for (int f = 0; f < n; f++) {
        memcpy(items[f].pts[0], left_points + (size_t)f * LANE_PTS * 2, sizeof(items[f].pts[0]));
        memcpy(items[f].pts[1], right_points + (size_t)f * LANE_PTS * 2, sizeof(items[f].pts[1]));
        items[f].valid[0] = left_valid[f] != 0;
        items[f].valid[1] = right_valid[f] != 0;
    }
    CudaEvent e0, e1;
    auto launch = [&](uint8_t *d_frames, uint8_t *) {
        if (device_ms) { e0.create(); e1.create(); cudaEventRecord(e0, st); }
        cudaMemcpyAsync(d, h, item_bytes, cudaMemcpyHostToDevice, st);
        LaneSrc src{(const char *)d, sizeof(LaneItem), {offsetof(LaneItem, pts), offsetof(LaneItem, pts) + sizeof(items[0].pts[0])},
                    {offsetof(LaneItem, valid), offsetof(LaneItem, valid) + 4}, 4};
        const int rc = launch_lanes(who, d_frames, src, n, height, width, fill_lane, st, device);
        if (device_ms) cudaEventRecord(e1, st);
        return rc;
    };
    const int rc = draw_frames(who, frames, on_device, (size_t)n * height * width * 3, device, st, false, launch);
    if (rc == LANE_OK && device_ms) cudaEventElapsedTime(device_ms, e0, e1);
    return rc;
}

extern "C" int lane_draw_lanes_records(uint8_t *frames_dev, int n, int height, int width, const lane_record *records_dev,
                                       int fill_lane, int device, void *cuda_stream)
{
    constexpr const char *who = "lane_draw_lanes_records";
    if (!frames_dev || !records_dev || n < 1 || height < 1 || width < 1) return lane_api_fail(LANE_ERR_INVALID, who, "bad arguments");
    if (height > 32767 || width > 32767) return lane_api_fail(LANE_ERR_UNSUPPORTED, who, "frame larger than 32767 px");
    if (int rc = lane_api_device(who, device)) return rc;
    LaneSrc src{(const char *)records_dev, sizeof(lane_record),
                {offsetof(lane_record, side) + offsetof(lane_side, points), offsetof(lane_record, side) + sizeof(lane_side) + offsetof(lane_side, points)},
                {offsetof(lane_record, side) + offsetof(lane_side, valid), offsetof(lane_record, side) + sizeof(lane_side) + offsetof(lane_side, valid)}, 4};
    return launch_lanes(who, frames_dev, src, n, height, width, fill_lane, (cudaStream_t)cuda_stream, device);
}

extern "C" int lane_generate_frames(uint8_t *frames, int on_device, int n, int height, int width, int64_t frame_count0,
                                    int device, void *cuda_stream, float *device_ms)
{
    constexpr const char *who = "lane_generate_frames";
    if (!frames || n < 1 || height < 1 || width < 1 || frame_count0 < 0) return lane_api_fail(LANE_ERR_INVALID, who, "bad arguments");
    if (height > 32767 || width > 32767) return lane_api_fail(LANE_ERR_UNSUPPORTED, who, "frame larger than 32767 px");
    if (int rc = lane_api_device(who, device)) return rc;
    return draw_driver(who, frames, on_device, n, height, width, device, (cudaStream_t)cuda_stream, device_ms,
                       [&](Builder &b, int f, const char **) {
                           build_generator_frame(b, frame_count0 + f);
                           return true;
                       },
                       true);
}
