// K1F: the fused edge kernel -- BGR -> gray -> 5x5 binomial blur -> histogram -> Sobel -> |dx|+|dy| -> sector NMS,
// one pass over the frames, nothing but bit-planes and a sparse byte plane written back.
//
// Replaces cv2.cvtColor(BGR2GRAY) + cv2.GaussianBlur((5,5),0) (lane_detector.py:69,72), the counting half of np.median
// (:79) and the gradient / non-maximum-suppression half of cv2.Canny (:83); arithmetic per SURVEY.md A.1-A.4.
//
// Why it can be one pass although the Canny thresholds depend on the median of the WHOLE blurred frame: non-maximum
// suppression does not depend on the thresholds at all (a pixel survives iff its magnitude beats its two neighbours
// along the gradient), only the final "m > low" / "m > high" tests do.  The kernel therefore emits, per pixel,
//   K  bit-plane  [H][W/32] : pixel survived NMS (and m > pre, see below)
//   V  byte plane [H][W]    : min(m, 256) - 1 for the survivors only (other bytes are never written or read)
// and the hysteresis kernel (k2_cluster.cu), which already needs the median, turns K/V into the candidate / strong
// planes with two byte compares (m > t  <=>  V >= t for t in 0..255) while it loads its band.  The blurred plane --
// the only full-resolution intermediate of the round-1 design (1 B/px written, 1 B/px read back) -- never exists.
//
// `pre` is a per-frame magnitude floor that keeps the exact sector test sparse: evaluating tan(22.5) sector logic on
// every pixel with a non-zero gradient (a third of a generator frame, all of a noisy one) would cost more than
// everything else together, whereas pixels with m <= low can never become edges.  low is not known yet, so pre comes
// from a sampled estimate of the median (k1_probe: 4096 gray samples per frame, pre = 7/8 of the low it implies).
// K is exact for every pixel with m > pre; the hysteresis kernel computes the true low and, if low < pre (the estimate
// was too optimistic), flags the frame, and the frame is redone with pre = low (launch_fused_edge_redo): results never
// depend on the estimate, only the time does.
//
// Data path (one warp = one 512-px column strip, 16 px per lane, rolling down a band of rows; warps pull (frame, band,
// strip) tasks from a global counter):
//   gray: 2 IDP2A per pixel straight off the interleaved BGR words, packed as u16x2 pairs (gray16)
//   vertical [1 4 6 4 1] as four chained pair-adds ([1 1]^4) on the packed pairs; horizontal pass: neighbours' edge pairs
//     by two shuffles, odd alignments by PRMT, +128 >> 8 folded into the byte pick
//   Sobel on the blurred row while it is still in registers: h1 = B(x+1) - B(x-1), h2 = B(x-1) + 2B(x) + B(x+1) per row,
//     dx = h1(r-1) + 2 h1(r) + h1(r+1), dy = h2(r+1) - h2(r-1) down the column, all as exact packed f16x2 (every value
//     is an integer below 2048 in units of 2^-24, where binary16 is exact and its bit pattern is the integer)
//   M, dx, dy of the last rows: per-warp shared-memory ring (16-bit), candidates = packed compare M > pre
//   NMS: the candidates of a row are spread over the 32 lanes through a small shared queue (an edge crossing the strip
//     puts its 3-4 candidate pixels into ONE lane's 16-px span; walking them in that lane would serialise the warp),
//     each lane does the TG22 sector test and the asymmetric 3x3 comparison for its share and ORs survivors into a
//     per-row bit string; fifteen lanes store the row's K words, survivors' V bytes go out as single byte stores
//   histogram: a per-warp table of 32-bit counters (shared-memory atomics), with a one-update fast path for lanes whose
//     sixteen blurred pixels are all equal (sky, asphalt)
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <type_traits>

#include <cuda_fp16.h>

#include "lane_common.cuh"

namespace {

constexpr int SPX = 16;                 // pixels per lane
constexpr int STRIP_OUT = 30 * SPX;     // 480 output pixels per warp (lanes 0 and 31 are halo providers)
constexpr int FWARPS = 4;               // warps per CTA
// CTAs per SM: 3 leaves 168 registers per thread.  Measured on B200, 256 x 1080p: 3 -> 0.74 ms, 4 -> 0.88 ms (at 128
// registers the spills cost more than four more warps hide).
constexpr int FCTAS = 3;
constexpr int RS = 512 + 16;            // M ring row stride in u16 (8 px of padding either side)

// per-warp shared memory (bytes)
constexpr int SM_TAB = 0;                          // [256] u32      histogram of the task (shared-memory atomics)
constexpr int SM_M = SM_TAB + 256 * 4;             // [3][RS] u16    magnitude ring
constexpr int SM_DX = SM_M + 3 * RS * 2;           // [2][512] u16   dx of rows s, s-1 (f16 sign-magnitude)
constexpr int SM_DY = SM_DX + 2 * 512 * 2;         // [2][512] u16
constexpr int SM_Q = SM_DY + 2 * 512 * 2;          // [512] u16      candidate queue of one row
constexpr int SM_KB = SM_Q + 512 * 2;              // [16] u32       K bits of one row (word w = px 32w .. 32w+31 of the strip)
constexpr int SM_QN = SM_KB + 16 * 4;              // u32            running count of queued candidates (never reset)
constexpr int SM_WARP = SM_QN + 16;                // 9392
static_assert(SM_WARP % 16 == 0, "per-warp block must keep 16-byte alignment");

__device__ __forceinline__ uint32_t dp2a_lo(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t d;
    asm("dp2a.lo.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ uint32_t dp2a_hi(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t d;
    asm("dp2a.hi.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ uint32_t h2add(uint32_t a, uint32_t b)
{
    uint32_t d;
    asm("add.f16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
    return d;
}
__device__ __forceinline__ uint32_t h2sub(uint32_t a, uint32_t b)
{
    uint32_t d;
    asm("sub.f16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
    return d;
}
__device__ __forceinline__ uint32_t h2abs_sum(uint32_t a, uint32_t b)   // |a| + |b|
{
    uint32_t d;
    asm("{\n\t.reg .b32 ta, tb;\n\tabs.f16x2 ta, %1;\n\tabs.f16x2 tb, %2;\n\tadd.f16x2 %0, ta, tb;\n\t}" : "=r"(d) : "r"(a), "r"(b));
    return d;
}
__device__ __forceinline__ uint32_t h2fma2(uint32_t a, uint32_t b)   // 2*a + b
{
    uint32_t d;
    asm("fma.rn.f16x2 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(0x40004000u), "r"(b));
    return d;
}
__device__ __forceinline__ uint4 ldg_stream(const uint4 *p)
{
    uint4 r;
    asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

// 16 interleaved BGR pixels (12 words) -> 8 packed u16x2 gray pairs (Q16 coefficients = 2x the Q15 ones, so the rounded
// value lands byte-aligned in bits 16..23 of each sum)
__device__ __forceinline__ void gray16(const uint32_t (&w)[12], uint32_t (&g)[8])
{
    constexpr uint32_t CB = 2 * 3735, CG = 2 * 19235, CR = 2 * 9798, RND = 1u << 15;
    constexpr uint32_t KBG = CB | (CG << 16), KR0 = CR, K0B = CB << 16, KGR = CG | (CR << 16);
#pragma unroll
    for (int q = 0; q < 4; q++) {       // 4 pixels per 3 words
        const uint32_t w0 = w[3 * q], w1 = w[3 * q + 1], w2 = w[3 * q + 2];
        uint32_t s0 = dp2a_hi(KR0, w0, dp2a_lo(KBG, w0, RND));   // B0 G0 R0 | .
        uint32_t s1 = dp2a_lo(KGR, w1, dp2a_hi(K0B, w0, RND));   // . . . B1 | G1 R1
        uint32_t s2 = dp2a_lo(KR0, w2, dp2a_hi(KBG, w1, RND));   // . . B2 G2 | R2
        uint32_t s3 = dp2a_hi(KGR, w2, dp2a_lo(K0B, w2, RND));   // . B3 G3 R3
        g[2 * q] = __byte_perm(s0, s1, 0x7632);
        g[2 * q + 1] = __byte_perm(s2, s3, 0x7632);
    }
}

// NMS of one row for the candidates queued by the warp (called only for rows that have candidates).
// Both loops have WARP-UNIFORM trip counts taken from redux instructions (max / sum of the lanes' candidate counts), with
// the per-lane work predicated inside.  That is deliberate: with per-lane trip counts (or a count read back from shared
// memory) ptxas can no longer prove that the warp is converged in the rest of the row step, guards every shuffle there
// with a BRA.DIV fallback path and pays ~60 register moves per row to keep the fallback's register layout.
// Returns (K word of this lane's slot in the row's bit string, new queue base).
__device__ __noinline__ uint2 nms_row(uint32_t cand, uint32_t qbase, uint8_t *ws, int sa, int sb, int sc, int parity,
                                      uint8_t *vrow)
{
    const int lane = threadIdx.x & 31;
    uint16_t *Mring = reinterpret_cast<uint16_t *>(ws + SM_M) + 8;
    const uint16_t *dxp = reinterpret_cast<uint16_t *>(ws + SM_DX) + parity * 512;
    const uint16_t *dyp = reinterpret_cast<uint16_t *>(ws + SM_DY) + parity * 512;
    uint16_t *queue = reinterpret_cast<uint16_t *>(ws + SM_Q);
    uint32_t *kbits = reinterpret_cast<uint32_t *>(ws + SM_KB);
    uint32_t *qn = reinterpret_cast<uint32_t *>(ws + SM_QN);
    // spread the row's candidates over the lanes
    const uint32_t cnt0 = (uint32_t)__popc(cand);
    {
        const uint32_t cnt = cnt0;
        uint32_t at = 0;
        if (cand) at = atomicAdd(qn, cnt) - qbase;
        const uint32_t xb = SPX * lane;
        const uint32_t most = __reduce_max_sync(0xffffffffu, cnt);      // warp-uniform trip count
        for (uint32_t k = 0; k < most; k++) {
            if (cand) {
                const int p = __ffs(cand) - 1;
                cand &= cand - 1;
                queue[at++] = (uint16_t)(xb + p);
            }
        }
    }
    __syncwarp();                                          // queue, M row s and dx/dy rows are visible to every lane
    // the counter only ever grows (no reset, hence no reset race): this row's entries are [qbase, *qn)
    const uint32_t total = __reduce_add_sync(0xffffffffu, cnt0), qend = qbase + total;
    const uint16_t *Ma = Mring + sa, *Mb = Mring + sb, *Mc = Mring + sc;
    for (uint32_t base = 0; base < total; base += 32) {
        const uint32_t i = base + lane;
        if (i >= total) continue;
        const uint32_t x = queue[i];
        const int m = Mb[x];
        const uint32_t xr = dxp[x], yr = dyp[x];
        const int a = (int)(xr & 0x7FFFu), b = (int)(yr & 0x7FFFu);
        const int tg22x = a * 13573, ay = b << 15;
        const uint16_t *p1, *p2;
        int ge;                                            // second comparison is >= for the axis-aligned sectors
        if (ay < tg22x) { p1 = Mb + x - 1; p2 = Mb + x + 1; ge = 1; }                    // horizontal gradient
        else if (ay > tg22x + (a << 16)) { p1 = Ma + x; p2 = Mc + x; ge = 1; }             // vertical
        else {                                             // diagonal: along (+1,+1) when the signs agree
            const int d = ((xr ^ yr) & 0x8000u) ? 1 : -1;
            p1 = Ma + x + d; p2 = Mc + x - d; ge = 0;
        }
        const int n1 = *p1, n2 = *p2;
        if (m > n1 && m + ge > n2) {
            const uint32_t xs = x - SPX;                   // pixel inside the strip's 480 outputs
            atomicOr(&kbits[xs >> 5], 1u << (xs & 31));
            vrow[xs] = (uint8_t)(min(m, 256) - 1);
        }
    }
    __syncwarp();                                          // all survivors are in kbits; ring slot sa is free again
    uint32_t kw = 0;
    if (lane < 16) {
        kw = kbits[lane];
        kbits[lane] = 0;
    }
    return make_uint2(kw, qend);
}

struct FusedArgs {
    const uint8_t *frames;         // [n][H][W][3]
    const int *frame_list;         // redo pass: indices of the frames to process (null = 0..n-1)
    const int *n_list;             // redo pass: number of entries in frame_list (device memory)
    uint32_t *hist;                // [n][256]; not touched in the redo pass (it is final already)
    const int *pre;                // [n] magnitude floor of the frame
    // first pass: the warp that finishes a frame last turns its histogram into the Canny thresholds
    int *frame_done;               // [n] tasks of the frame finished so far (zeroed by the launcher)
    const uint8_t *lut_low, *lut_high;
    int4 *thr;                     // [n] (2 * median, low, high, floor used)
    int *pre_redo, *redo_list, *redo_count, *redo_flag;   // frames whose true low is below the floor: redone with pre = low
    uint32_t *k_bits;              // [n][H][WW]
    uint8_t *v_plane;              // [n][H][W]
    uint8_t *blur_dbg;             // [n][H][W] or null: the blurred plane, for the verification taps only
    int *task_counter;
    int n_frames, H, W, WW;
    int band_rows, tail_frames, tail_rows;
};

__global__ void __launch_bounds__(FWARPS * 32, FCTAS) k1_fused(FusedArgs A)
{
    extern __shared__ __align__(128) uint8_t fsm[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint8_t *ws = fsm + wid * SM_WARP;
    uint32_t *tab = reinterpret_cast<uint32_t *>(ws + SM_TAB);
    uint16_t *Mring = reinterpret_cast<uint16_t *>(ws + SM_M) + 8;     // + slot * RS
    uint16_t *DXr = reinterpret_cast<uint16_t *>(ws + SM_DX), *DYr = reinterpret_cast<uint16_t *>(ws + SM_DY);
    uint32_t *kbits = reinterpret_cast<uint32_t *>(ws + SM_KB);
    uint32_t *qn = reinterpret_cast<uint32_t *>(ws + SM_QN);
    const int H = A.H, W = A.W, WW = A.WW;
    const bool redo = A.frame_list != nullptr;
    const int n_frames = redo ? *A.n_list : A.n_frames;
    const int tail_frames = redo ? 0 : A.tail_frames;
    {   // zero this warp's K bits and queue length
        if (lane < 16) kbits[lane] = 0;
        if (lane == 0) *qn = 0;
    }
    __syncwarp();
    uint32_t qbase = 0;                                   // value of *qn when the current row's queue starts (warp-uniform)
    const int n_strips = (W + STRIP_OUT - 1) / STRIP_OUT;
    const int n_bands = (H + A.band_rows - 1) / A.band_rows, n_bands_t = (H + A.tail_rows - 1) / A.tail_rows;
    const int n_main = (n_frames - tail_frames) * n_bands * n_strips;
    const int n_tasks = n_main + tail_frames * n_bands_t * n_strips;
    const size_t frame_px = (size_t)H * W;
    const uint32_t xb = SPX * lane;                       // first pixel of this lane in strip coordinates
    const uint32_t hbase = smem_u32(tab);

    for (;;) {
        int task = 0;
        if (lane == 0) task = atomicAdd(A.task_counter, 1);
        task = __shfl_sync(0xffffffffu, task, 0);
        if (task >= n_tasks) break;
        const bool tail = task >= n_main;
        const int tt = tail ? task - n_main : task, nb = tail ? n_bands_t : n_bands, br = tail ? A.tail_rows : A.band_rows;
        const int strip = tt % n_strips;
        const int band = (tt / n_strips) % nb;
        const int fi = tt / (n_strips * nb) + (tail ? n_frames - tail_frames : 0);
        const int f = redo ? A.frame_list[fi] : fi;
        const int q0 = band * br, q1 = min(q0 + br, H);
        const int xl = strip * STRIP_OUT - SPX + SPX * lane;          // first pixel of this lane in the frame
        const bool in_img = xl >= 0 && xl < W;
        const bool is_out = in_img && lane >= 1 && lane <= 30;
        const bool left_edge = xl == 0, right_edge = xl + SPX == W;
        const uint8_t *src = A.frames + f * frame_px * 3 + (size_t)max(xl, 0) * 3;
        uint8_t *bdst = A.blur_dbg ? A.blur_dbg + f * frame_px + max(xl, 0) : nullptr;
        const bool dbg_store = bdst != nullptr && is_out;
        uint8_t *vrow = A.v_plane + f * frame_px + (size_t)q0 * W + strip * STRIP_OUT;      // row n of V: + (x - 16)
        const int word0 = strip * (STRIP_OUT / 32);
        uint32_t *krow = A.k_bits + ((size_t)f * H + q0) * WW + word0 + lane;                // row n of K (lanes 0..14)
        const bool k_writer = lane < STRIP_OUT / 32 && word0 + lane < WW;
        const uint32_t pre = (uint32_t)A.pre[f];
        const uint32_t pre2 = pre | (pre << 16);
        const uint32_t own_mask = is_out ? 0xFFFFu : 0u;

        // blur column-filter state, two generations deep (slots alternate by row, the row loop is unrolled by two)
        uint32_t sg[2][8], s1[2][8], s2[2][8], s3[2][8];
        // Sobel column state: h1 and T1 = h1(r-1) + h1(r) of the previous row, h2 of the previous two rows
        uint32_t h1s[2][8], T1s[2][8], h2s[2][8];
#pragma unroll
        for (int j = 0; j < 8; j++) {
            sg[0][j] = sg[1][j] = s1[0][j] = s1[1][j] = s2[0][j] = s2[1][j] = s3[0][j] = s3[1][j] = 0;
            h1s[0][j] = h1s[1][j] = T1s[0][j] = T1s[1][j] = h2s[0][j] = h2s[1][j] = 0;
        }
        if (!redo) {
#pragma unroll
            for (int b = 0; b < 8; b++) tab[b * 32 + lane] = 0;
        }
        if (!in_img) {                                    // the magnitude plane has a zero border beyond the image
#pragma unroll
            for (int sl = 0; sl < 3; sl++) {
                uint4 *z = reinterpret_cast<uint4 *>(Mring + sl * RS + xb);
                z[0] = make_uint4(0, 0, 0, 0); z[1] = make_uint4(0, 0, 0, 0);
            }
        }
        uint32_t cand_prev = 0;                           // candidates of the row whose NMS runs next
        int sa = 0, sb = RS, sc = 2 * RS;                 // ring slots of M rows s-2, s-1, s

        uint32_t w[12];
        auto load_row = [&](int y) {
            // BORDER_REFLECT_101 for the gray rows above / below the frame (|y|, then mirrored at the bottom)
            const int ya = abs(y), yy = min(ya, 2 * H - 2 - ya);
            if (in_img) {
                const uint4 *p = reinterpret_cast<const uint4 *>(src + (uint32_t)(yy * W) * 3u);
                uint4 a = ldg_stream(p), b = ldg_stream(p + 1), c = ldg_stream(p + 2);
                w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
                w[8] = c.x; w[9] = c.y; w[10] = c.z; w[11] = c.w;
            }
        };
#pragma unroll
        for (int j = 0; j < 12; j++) w[j] = 0;
        const int y_first = q0 - 4, y_last = q1 + 3;      // gray rows this band reads
        load_row(y_first);

        // pipeline fill: the first four gray rows only feed the vertical filter
        auto fill_step = [&](auto slot, int y) {
            constexpr int c = decltype(slot)::value, o = c ^ 1;
            gray16(w, sg[c]);
            load_row(y + 1);
#pragma unroll
            for (int j = 0; j < 8; j++) {
                s1[c][j] = h2add(sg[c][j], sg[o][j]);
                s2[c][j] = h2add(s1[c][j], s1[o][j]);
                s3[c][j] = h2add(s2[c][j], s2[o][j]);
            }
        };
        // One row of the steady state.  No persistent array is assigned under a condition here (the frame borders are
        // patched in shared memory by a rare branch below): every conditional assignment to the column state costs a
        // block of register moves per row once the compiler has to merge the two versions.
        auto row_step = [&](auto slot, int y) {
            constexpr int c = decltype(slot)::value, o = c ^ 1;
            gray16(w, sg[c]);
            if (y < y_last) load_row(y + 1);             // prefetch the next row behind the arithmetic
            uint32_t V[8];
#pragma unroll
            for (int j = 0; j < 8; j++) {                // [1 1]^4 down the column; stages < 2048 as exact add.f16x2
                s1[c][j] = h2add(sg[c][j], sg[o][j]);
                s2[c][j] = h2add(s1[c][j], s1[o][j]);
                s3[c][j] = h2add(s2[c][j], s2[o][j]);
                V[j] = s3[c][j] + s3[o][j];
            }
            const int r = y - 2;                          // V is the column sum of blurred row r
            // ---- horizontal [1 4 6 4 1]
            uint32_t Bp[8];                               // blurred row r as zero-interleaved pairs (f16x2 integers)
            {
                uint32_t L7 = __shfl_up_sync(0xffffffffu, V[7], 1);
                uint32_t R0 = __shfl_down_sync(0xffffffffu, V[0], 1);
                if (left_edge) L7 = __byte_perm(V[1], V[0], 0x7610);     // (x=-2,-1) := (x=2, 1)
                if (right_edge) R0 = __byte_perm(V[7], V[6], 0x7610);    // (x=W, W+1) := (x=W-2, W-3)
                uint32_t O[9];
                O[0] = __byte_perm(L7, V[0], 0x5432);
#pragma unroll
                for (int j = 1; j < 8; j++) O[j] = __byte_perm(V[j - 1], V[j], 0x5432);
                O[8] = __byte_perm(V[7], R0, 0x5432);
                uint32_t Hs[8];
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    const uint32_t vm = j == 0 ? L7 : V[j - 1], vp = j == 7 ? R0 : V[j + 1];
                    Hs[j] = vm + vp + 0x00800080u + 4u * (O[j] + O[j + 1]) + 6u * V[j];
                    Bp[j] = __byte_perm(Hs[j], 0, 0x4341);               // (Hs >> 8) per half
                }
                if (r >= q0 && r < q1) {                  // rows this band owns: histogram (and the debug plane)
                    uint4 ov;
                    ov.x = __byte_perm(Hs[0], Hs[1], 0x7531);
                    ov.y = __byte_perm(Hs[2], Hs[3], 0x7531);
                    ov.z = __byte_perm(Hs[4], Hs[5], 0x7531);
                    ov.w = __byte_perm(Hs[6], Hs[7], 0x7531);
                    if (dbg_store) *reinterpret_cast<uint4 *>(bdst + (uint32_t)r * (uint32_t)W) = ov;
                    if (!redo) {
                        // Histogram of the task in a per-warp table of 32-bit counters, updated with shared-memory
                        // atomics (fire and forget; 1 KB per warp instead of 8 KB of per-lane byte counters, which is what
                        // lets 16 warps share an SM).  A lane whose sixteen pixels are equal (flat sky / asphalt) adds 16
                        // once; when the whole 480-px row of the strip is one value, one lane adds it all.
                        const bool flat = ov.x == ov.y && ov.z == ov.w && ov.x == ov.z && ov.x == __byte_perm(ov.x, 0, 0);
                        const uint32_t v0 = __shfl_sync(0xffffffffu, ov.x, 1);
                        const unsigned out_lanes = __ballot_sync(0xffffffffu, is_out);
                        if (__all_sync(0xffffffffu, !is_out || (flat && ov.x == v0))) {
                            if (lane == 1) atomicAdd(&tab[v0 & 0xFFu], 16u * (uint32_t)__popc(out_lanes));
                        } else if (__all_sync(0xffffffffu, flat || !is_out)) {
                            if (is_out) atomicAdd(&tab[ov.x & 0xFFu], 16u);
                        } else if (is_out) {
                            const uint32_t ow[4] = {ov.x, ov.y, ov.z, ov.w};
#pragma unroll
                            for (int q = 0; q < 4; q++) {
#pragma unroll
                                for (int k = 0; k < 4; k++) {
                                    // counter address = base + 4 * byte k of the word, in one dot-product instruction
                                    const uint32_t addr = __dp4a(ow[q], 0x4u << (8 * k), hbase);
                                    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(addr), "r"(1u) : "memory");
                                }
                            }
                        }
                    }
                }
            }
            // ---- Sobel, arrival of blurred row r: forms the gradient of row s = r - 1
            const int s = r - 1;
            uint32_t dx[8], dy[8], Mw[8], cand_new;
            {
                uint32_t BL = __shfl_up_sync(0xffffffffu, Bp[7], 1), BR = __shfl_down_sync(0xffffffffu, Bp[0], 1);
                if (left_edge) BL = __byte_perm(Bp[0], 0, 0x1010);       // x=-1 := x=0 (BORDER_REPLICATE)
                if (right_edge) BR = __byte_perm(Bp[7], 0, 0x3232);      // x=W := x=W-1
                uint32_t Bo[9];                                            // odd-aligned pairs (B(2j-1), B(2j))
                Bo[0] = __byte_perm(BL, Bp[0], 0x5432);
#pragma unroll
                for (int j = 1; j < 8; j++) Bo[j] = __byte_perm(Bp[j - 1], Bp[j], 0x5432);
                Bo[8] = __byte_perm(Bp[7], BR, 0x5432);
                uint32_t acc = 0;
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    h1s[c][j] = h2sub(Bo[j + 1], Bo[j]);                   // B(x+1) - B(x-1)
                    const uint32_t h2old = h2s[c][j];                      // h2 of row r - 2
                    h2s[c][j] = h2fma2(Bp[j], h2add(Bo[j], Bo[j + 1]));    // B(x-1) + 2 B(x) + B(x+1)
                    T1s[c][j] = h2add(h1s[o][j], h1s[c][j]);
                    dx[j] = h2add(T1s[o][j], T1s[c][j]);                   // h1(s-1) + 2 h1(s) + h1(s+1)
                    dy[j] = h2sub(h2s[c][j], h2old);                       // h2(s+1) - h2(s-1)
                    Mw[j] = h2abs_sum(dx[j], dy[j]);
                    const uint32_t gt = __hgt2_mask(*reinterpret_cast<const __half2 *>(&Mw[j]),
                                                    *reinterpret_cast<const __half2 *>(&pre2));   // 0xFFFF per half: M > pre
                    acc |= gt & ((1u << (2 * j)) | (1u << (2 * j + 17)));
                }
                cand_new = (acc | (acc >> 16)) & own_mask;
            }
            uint4 *mrow = reinterpret_cast<uint4 *>(Mring + sc + xb);
            uint4 *xrow = reinterpret_cast<uint4 *>(DXr + (s & 1) * 512 + xb);
            uint4 *yrow = reinterpret_cast<uint4 *>(DYr + (s & 1) * 512 + xb);
            if (s <= 0 || s >= H - 1) {
                // Frame borders (warp-uniform, two rows per frame).  The blurred plane is extended by BORDER_REPLICATE
                // (row -1 := row 0, row H := row H-1) while the rows the filter state saw there came from the reflected
                // gray rows, and the magnitude is zero outside the frame: redo this row's gradient from the state.
                uint32_t acc = 0;
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    uint32_t ex, ey;
                    if (s == 0) {                          // h1(-1) = h1(0), h2(-1) = h2(0)
                        ex = h2add(T1s[c][j], h2add(h1s[o][j], h1s[o][j]));
                        ey = h2sub(h2s[c][j], h2s[o][j]);
                    } else {                               // s == H-1: h1(H) = h1(H-1), h2(H) = h2(H-1); h2(H-2) = h2new - dy
                        ex = h2add(T1s[o][j], h2add(h1s[o][j], h1s[o][j]));
                        ey = h2sub(h2s[o][j], h2sub(h2s[c][j], dy[j]));
                    }
                    uint32_t em = h2abs_sum(ex, ey);
                    if (s < 0 || s >= H) { ex = 0; ey = 0; em = 0; }
                    const uint32_t gt = __hgt2_mask(*reinterpret_cast<const __half2 *>(&em),
                                                    *reinterpret_cast<const __half2 *>(&pre2));
                    acc |= gt & ((1u << (2 * j)) | (1u << (2 * j + 17)));
                    dx[j] = ex; dy[j] = ey; Mw[j] = em;
                }
                cand_new = (acc | (acc >> 16)) & own_mask;
                if (in_img) {
                    mrow[0] = make_uint4(Mw[0], Mw[1], Mw[2], Mw[3]); mrow[1] = make_uint4(Mw[4], Mw[5], Mw[6], Mw[7]);
                }
                xrow[0] = make_uint4(dx[0], dx[1], dx[2], dx[3]); xrow[1] = make_uint4(dx[4], dx[5], dx[6], dx[7]);
                yrow[0] = make_uint4(dy[0], dy[1], dy[2], dy[3]); yrow[1] = make_uint4(dy[4], dy[5], dy[6], dy[7]);
            } else {
                if (in_img) {
                    mrow[0] = make_uint4(Mw[0], Mw[1], Mw[2], Mw[3]); mrow[1] = make_uint4(Mw[4], Mw[5], Mw[6], Mw[7]);
                }
                if (cand_new) {                            // only candidates' gradients are ever read back
                    xrow[0] = make_uint4(dx[0], dx[1], dx[2], dx[3]); xrow[1] = make_uint4(dx[4], dx[5], dx[6], dx[7]);
                    yrow[0] = make_uint4(dy[0], dy[1], dy[2], dy[3]); yrow[1] = make_uint4(dy[4], dy[5], dy[6], dy[7]);
                }
            }
            // ---- NMS of row n = s - 1 (M rows n-1, n, n+1 in ring slots sa, sb, sc)
            const int n = s - 1;
            if (n >= q0) {
                uint32_t kw = 0;
                if (__any_sync(0xffffffffu, cand_prev != 0)) {
                    const uint2 res = nms_row(cand_prev, qbase, ws, sa, sb, sc, n & 1, vrow);
                    kw = res.x; qbase = res.y;
                }
                if (k_writer) *krow = kw;
                krow += WW; vrow += W;
            }
            cand_prev = cand_new;
            const int t = sa; sa = sb; sb = sc; sc = t;
        };
        {
            int y = y_first;
            fill_step(std::integral_constant<int, 0>{}, y++);
            fill_step(std::integral_constant<int, 1>{}, y++);
            fill_step(std::integral_constant<int, 0>{}, y++);
            fill_step(std::integral_constant<int, 1>{}, y++);
            for (;;) {
                row_step(std::integral_constant<int, 0>{}, y);
                if (++y > y_last) break;
                row_step(std::integral_constant<int, 1>{}, y);
                if (++y > y_last) break;
            }
        }
        __syncwarp();
        if (!redo) {
#pragma unroll
            for (int b = 0; b < 8; b++)
                if (const uint32_t t = tab[b * 32 + lane]) atomicAdd(&A.hist[f * 256 + b * 32 + lane], t);
            // np.median + thresholds (lane_detector.py:79-81) once per frame, by whoever completes it
            __threadfence();
            int done = 0;
            if (lane == 0) done = atomicAdd(&A.frame_done[f], 1);
            done = __shfl_sync(0xffffffffu, done, 0);
            if (done == nb * n_strips - 1) {
                __threadfence();
                const int m2 = median_x2_warp(A.hist + f * 256, (long long)H * W, lane);
                int low = A.lut_low[m2], high = A.lut_high[m2];
                if (low > high) { const int t = low; low = high; high = t; }
                if (lane == 0) {
                    A.thr[f] = make_int4(m2, low, high, (int)pre);
                    const int again = low < (int)pre;      // the sampled floor was too high: K misses candidates
                    A.redo_flag[f] = again;
                    if (again) {
                        A.pre_redo[f] = low;
                        A.redo_list[atomicAdd(A.redo_count, 1)] = f;
                    }
                }
            }
        }
        __syncwarp();                                     // the table is zeroed again at the start of the next task
    }
}

// ---- k1_probe: a sampled estimate of the blurred frame's median -> the magnitude floor `pre` of k1_fused ----------
// 64 x 64 lattice of gray samples per frame (unblurred: an estimate is all that is needed), median by a 256-bin
// shared-memory histogram, low_est = lut_low[2 * median], pre = low_est - max(4, low_est / 8) clamped at 0.
__global__ void __launch_bounds__(256) k1_probe(const uint8_t *__restrict__ frames, const uint8_t *__restrict__ lut_low,
                                                int *__restrict__ pre, int H, int W, int forced)
{
    __shared__ uint32_t h[256];
    const int f = blockIdx.x, tid = threadIdx.x;
    if (forced >= 0) {                                    // test hook: a given floor for every frame (exercises the redo path)
        if (tid == 0) pre[f] = forced;
        return;
    }
    h[tid] = 0;
    __syncthreads();
    const uint8_t *src = frames + (size_t)f * H * W * 3;
    const int ny = min(H, 64), nx = min(W, 64);
    if (ny == 64 && nx == 64) {
        // sixteen samples per thread, every load issued before the first is used (the samples are DRAM misses); sample
        // (iy, ix) of the 64 x 64 lattice sits at the centre of its cell (32-bit arithmetic: sides are below 32768)
        uint32_t g[16];
#pragma unroll
        for (int u = 0; u < 16; u++) {
            const uint32_t i = tid + u * 256, iy = i >> 6, ix = i & 63u;
            const uint32_t y = ((2u * iy + 1u) * (uint32_t)H) >> 7, x = ((2u * ix + 1u) * (uint32_t)W) >> 7;
            const uint8_t *p = src + (y * (uint32_t)W + x) * 3u;
            g[u] = 3735u * __ldg(p) + 19235u * __ldg(p + 1) + 9798u * __ldg(p + 2);
        }
#pragma unroll
        for (int u = 0; u < 16; u++) atomicAdd(&h[(g[u] + (1u << 14)) >> 15], 1u);
    } else {                                              // frames smaller than the lattice: every row / column once
        for (int i = tid; i < ny * nx; i += 256) {
            const int iy = i / nx, ix = i - iy * nx;
            const int y = ((2 * iy + 1) * H) / (2 * ny), x = ((2 * ix + 1) * W) / (2 * nx);
            const uint8_t *p = src + ((size_t)y * W + x) * 3;
            atomicAdd(&h[(3735u * p[0] + 19235u * p[1] + 9798u * p[2] + (1u << 14)) >> 15], 1u);
        }
    }
    __syncthreads();
    if (tid == 0) {
        const int half = (ny * nx) / 2;
        int run = 0, med = 255;
        for (int v = 0; v < 256; v++) {
            run += (int)h[v];
            if (run > half) { med = v; break; }
        }
        const int low = lut_low[2 * med];
        pre[f] = max(0, low - max(4, low / 8));
    }
}

}  // namespace

bool lane_fused_edge_supported(int H, int W, const void *frames)
{
    return (W % 16 == 0) && H >= 16 && ((uintptr_t)frames % 16 == 0) && (size_t)H * W * 3 < ((size_t)1 << 32);
}

static void fused_config(int n, int H, int W, int *band_rows, int *tail_frames, int *tail_rows)
{
    const int sms = lane_sm_count();
    const int n_strips = (W + STRIP_OUT - 1) / STRIP_OUT, warps = sms * FCTAS * FWARPS;
    // Every band re-reads 8 halo rows (7 % at 108 rows), but a task is also the unit the warps run dry by at the end of
    // the kernel (a row takes a warp ~1 us): measured on B200 (256 x 1080p) 108-row bands with the last eighth of the
    // frames cut into bands a third as high beat both taller bands (135: +1 %, 270: +15 %) and a shorter graded tail
    // (n/16: +4 %).  Small batches get thinner bands so that every resident warp has at least two tasks.
    int br = H >= 540 ? 108 : (H >= 120 ? 60 : H);
    const long rows_per_warp = ((long)n * H * n_strips + 2 * warps - 1) / (2 * warps);
    br = (int)std::max(16L, std::min((long)br, rows_per_warp));
    int tf = n >= 16 ? n / 8 : 0;
    const int tr = std::max(16, br / 3);
    if (tr >= br) tf = 0;
    *band_rows = br; *tail_frames = tf; *tail_rows = tr;
}

static bool fused_launch(FusedArgs A, cudaStream_t st)
{
    static bool configured[LANE_MAX_DEVICES];
    if (!configured[lane_cur_device()]) {
        if (cudaFuncSetAttribute(k1_fused, cudaFuncAttributeMaxDynamicSharedMemorySize, FWARPS * SM_WARP) != cudaSuccess) {
            cudaGetLastError();
            return false;
        }
        configured[lane_cur_device()] = true;
    }
    cudaMemsetAsync(A.task_counter, 0, sizeof(int), st);
    k1_fused<<<lane_sm_count() * FCTAS, FWARPS * 32, FWARPS * SM_WARP, st>>>(A);
    return cudaPeekAtLastError() == cudaSuccess;
}

// First pass over frames 0..n-1: estimate the floors, then gray + blur + histogram + Sobel + NMS in one kernel.
bool launch_fused_edge(const uint8_t *frames, const uint8_t *lut_low, const uint8_t *lut_high, uint32_t *hist, int4 *thr,
                       int *pre, int *pre_redo, int *redo_list, int *redo_count, int *redo_flag, int *frame_done,
                       uint32_t *k_bits, uint8_t *v_plane, uint8_t *blur_dbg, int *task_counter, int n, int H, int W,
                       cudaStream_t st, int *launches)
{
    static const int forced = getenv("LANE_K1F_PRE") ? atoi(getenv("LANE_K1F_PRE")) : -1;
    cudaMemsetAsync(hist, 0, sizeof(uint32_t) * 256 * n, st);
    cudaMemsetAsync(frame_done, 0, sizeof(int) * n, st);
    cudaMemsetAsync(redo_count, 0, sizeof(int), st);
    k1_probe<<<n, 256, 0, st>>>(frames, lut_low, pre, H, W, forced);
    FusedArgs A{};
    A.frame_done = frame_done; A.lut_low = lut_low; A.lut_high = lut_high; A.thr = thr; A.pre_redo = pre_redo;
    A.redo_list = redo_list; A.redo_count = redo_count; A.redo_flag = redo_flag;
    A.frames = frames; A.frame_list = nullptr; A.n_list = nullptr; A.hist = hist; A.pre = pre; A.k_bits = k_bits;
    A.v_plane = v_plane; A.blur_dbg = blur_dbg; A.task_counter = task_counter;
    A.n_frames = n; A.H = H; A.W = W; A.WW = (W + 31) / 32;
    fused_config(n, H, W, &A.band_rows, &A.tail_frames, &A.tail_rows);
    if (!fused_launch(A, st)) { cudaGetLastError(); return false; }
    *launches += 2;
    return true;
}

// Redo pass: the frames the hysteresis kernel listed (true low below the floor used), with pre[f] = low[f] now exact.
bool launch_fused_edge_redo(const uint8_t *frames, const int *frame_list, const int *n_list, const int *pre,
                            uint32_t *k_bits, uint8_t *v_plane, uint8_t *blur_dbg, int *task_counter, int n, int H, int W,
                            cudaStream_t st, int *launches)
{
    FusedArgs A{};
    A.frames = frames; A.frame_list = frame_list; A.n_list = n_list; A.hist = nullptr; A.pre = pre; A.k_bits = k_bits;
    A.v_plane = v_plane; A.blur_dbg = blur_dbg; A.task_counter = task_counter;
    A.n_frames = n; A.H = H; A.W = W; A.WW = (W + 31) / 32;
    fused_config(n, H, W, &A.band_rows, &A.tail_frames, &A.tail_rows);
    A.tail_frames = 0;
    if (!fused_launch(A, st)) { cudaGetLastError(); return false; }
    *launches += 1;
    return true;
}
