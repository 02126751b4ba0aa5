// K2 (cluster form): thresholds + Sobel + NMS + double threshold + hysteresis + ROI compaction
// for one frame per thread-block cluster, bit-planes in (distributed) shared memory.
//
// Replaces np.median/low/high (lane_detector.py:79-81), cv2.Canny (:83), the ROI mask (:86-90) and the
// row-major nzloc scan of cv2.HoughLinesP (:94); arithmetic per SURVEY.md A.3/A.4.
//
//   cluster = G CTAs, CTA r owns a band of rows.  Per CTA:
//   phase 1  warps roll down 512-px column strips of the blurred plane (one 16-byte load per lane per
//            row).  Sobel and |dx|+|dy| run as packed f16x2 on the zero-interleaved bytes: every value
//            is an integer below 2048 in units of 2^-24, which binary16 (denormals included) holds
//            exactly and whose bit pattern IS the integer, so the result is bit-exact integer math at
//            two pixels per instruction.  Only pixels whose magnitude beats `low` (sparse) take the
//            scalar sector test (TG22 fixed point) and the 3x3 non-maximum test.  Candidate / strong
//            bits leave the registers as 32-px words into two bit-planes C and S in shared memory.
//   phase 2  hysteresis = S <- closure of S inside C under 8-connectivity: word-parallel dilation
//            (32 px per op), in-word flood by carry propagation, column-serial sweeps down and up,
//            __syncthreads_or convergence per CTA; bands exchange their boundary rows over DSMEM and
//            a cluster barrier until no band saw a change.
//   phase 3  edge bit-plane, edge count, ROI-masked bit-plane (the PPHT mask) and the row-major point
//            list (offsets by per-row popcounts, band bases exchanged over DSMEM).
#include <algorithm>
#include <cooperative_groups.h>
#include <cuda_fp16.h>
#include <stdio.h>
#include <stdlib.h>

#include "lane_common.cuh"
#include <type_traits>

namespace cg = cooperative_groups;

namespace {

constexpr int K2T = 256;
constexpr int SPX = 16;
constexpr int STRIP_OUT = 30 * SPX;

struct K2Args {
    const uint32_t *c_bits, *s_bits;   // [n][H][WW] candidate / strong planes (from k2a_sobel_nms or k2t_threshold)
    const int *skip_flag;              // [n] or null: frames waiting for the redo pass (fused path) are skipped
    const int *frame_list, *n_list;    // redo pass: the frames to process (null = all)
    const uint32_t *roi_bits;      // [R][roi_stride] ROI planes, each [H][WW]
    int *n_edges, *rounds, *n_points;
    uint32_t *points;              // [n][max_points]
    uint32_t *pmask_bits;          // [n][bh][WW]
    uint32_t *edge_bits;           // [n][H][WW]
    int H, W, WW, R;               // R = rows per band
    LaneGeom g;
    const int *roi_index;          // [n] ROI plane of each frame, or null: every frame uses plane 0
    size_t roi_stride;             // words between planes (0 with a null roi_index)
};

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
__device__ __forceinline__ uint32_t h2abs_sum(uint32_t a, uint32_t b)   // |a| + |b| (the abs folds into HADD2's operand modifiers)
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

// Sobel + NMS for one (strip, row range) task; writes the C/S words of rows [q0,q1) of the frame's planes.
//
// Dense part (every pixel, two per instruction): column sums T(c) = B(c) + B(c+1) give the Sobel column filters as
// T(c-1) + T(c) and T(c) - T(c-1); the row loop is unrolled by two with compile-time slots so the two generations of
// B and T rotate by renaming.  The magnitude row and the signed gradients go to a per-warp shared-memory ring (3 rows
// of M, 2 of dx/dy) as 16-bit values, and a packed compare gives the 16-bit candidate mask of the lane.
// Sparse part (candidates only, one row later when the row below exists): every lane walks the set bits of its own
// mask and does the sector test (TG22 fixed point) and the 3x3 non-maximum test with plain 16-bit loads from the
// ring -- neighbours in other lanes' columns are just addresses, no shuffles or compile-time pixel indices.
constexpr int K2A_RS = 512 + 16;                         // M ring row stride in u16 (8 px of padding either side)
constexpr int K2A_WSM = 3 * K2A_RS + 4 * 512;            // u16 per warp: M[3][RS] | DX[2][512] | DY[2][512]

__device__ __forceinline__ void canny_rows(int H, int W, int WW, const uint8_t *blur_f, int strip, int q0, int q1,
                                           uint32_t *Cw, uint32_t *Sw, int lane, int low, int high, uint16_t *wsm)
{
    const int xl = strip * STRIP_OUT - SPX + SPX * lane;
    const bool in_img = xl >= 0 && xl < W;
    const bool left_edge = xl == 0, right_edge = xl + SPX == W;
    const uint8_t *src = blur_f + max(xl, 0);
    const int word = strip * (STRIP_OUT / 32) + ((lane - 1) >> 1);
    const bool writer = (lane & 1) && lane <= 29 && in_img && word < WW;
    const uint32_t low2 = (uint32_t)low | ((uint32_t)low << 16);
    const uint32_t xb = SPX * lane;
    const uint32_t own_mask = (lane >= 1 && lane <= 30 && in_img) ? 0xFFFFu : 0u;   // halo lanes only feed neighbours
    uint16_t *Mring = wsm + 8;                               // + slot * K2A_RS
    uint16_t *DXr = wsm + 3 * K2A_RS, *DYr = DXr + 2 * 512;  // + (row & 1) * 512

    uint32_t Bs[2][8], Ts[2][8];
    auto load_raw = [&](int y) {
        const uint32_t off = (uint32_t)min(max(y, 0), H - 1) * (uint32_t)W;          // BORDER_REPLICATE rows
        uint4 v = make_uint4(0, 0, 0, 0);
        if (in_img) v = __ldg(reinterpret_cast<const uint4 *>(src + off));
        return v;
    };
    auto unpack = [&](const uint4 &v, uint32_t (&b)[8]) {   // bytes -> zero-interleaved pairs (= f16x2 denormals)
        b[0] = __byte_perm(v.x, 0, 0x4140); b[1] = __byte_perm(v.x, 0, 0x4342);
        b[2] = __byte_perm(v.y, 0, 0x4140); b[3] = __byte_perm(v.y, 0, 0x4342);
        b[4] = __byte_perm(v.z, 0, 0x4140); b[5] = __byte_perm(v.z, 0, 0x4342);
        b[6] = __byte_perm(v.w, 0, 0x4140); b[7] = __byte_perm(v.w, 0, 0x4342);
    };
    if (!in_img) {                                         // zero magnitude beyond the image border, for the whole task
#pragma unroll
        for (int sl = 0; sl < 3; sl++) {
            uint4 *z = reinterpret_cast<uint4 *>(Mring + sl * K2A_RS + xb);
            z[0] = make_uint4(0, 0, 0, 0); z[1] = make_uint4(0, 0, 0, 0);
        }
    }
    unpack(load_raw(q0 - 2), Bs[0]);
    unpack(load_raw(q0 - 1), Bs[1]);
#pragma unroll
    for (int j = 0; j < 8; j++) Ts[1][j] = h2add(Bs[0][j], Bs[1][j]);       // T(q0-2)
    uint4 vnext = load_raw(q0);                         // row c+1 of the first step
    uint32_t out_idx = (uint32_t)q0 * WW + word;        // plane word of row n
    uint32_t cand_prev = 0;                             // candidates of row c-1
    int sa = 0, sb = K2A_RS, sc = 2 * K2A_RS;           // ring slots of rows c-2, c-1, c

    auto step = [&](auto slot, int c) {                 // c = row whose gradient is formed this step
        constexpr int k = decltype(slot)::value, o = k ^ 1;
        unpack(vnext, Bs[k]);                            // row c+1
        if (c < q1) vnext = load_raw(c + 2);             // prefetch the next step's row behind the arithmetic
        // the magnitude plane has a zero border: rows outside the frame give M = 0 (lanes outside the image never
        // store their M; their ring entries were zeroed once)
        const bool row_ok = c >= 0 && c < H;
        uint32_t cand_new;
        {
            uint32_t Sc[8], Dc[8];
#pragma unroll
            for (int j = 0; j < 8; j++) {
                Ts[k][j] = h2add(Bs[k][j], Bs[o][j]);            // T(c) = B(c+1) + B(c)
                Sc[j] = h2add(Ts[k][j], Ts[o][j]);               // column [1 2 1]
                Dc[j] = h2sub(Ts[k][j], Ts[o][j]);               // column [-1 0 1]
            }
            uint32_t SL = __shfl_up_sync(0xffffffffu, Sc[7], 1), SR = __shfl_down_sync(0xffffffffu, Sc[0], 1);
            uint32_t DL = __shfl_up_sync(0xffffffffu, Dc[7], 1), DR = __shfl_down_sync(0xffffffffu, Dc[0], 1);
            if (left_edge) { SL = __byte_perm(Sc[0], 0, 0x1010); DL = __byte_perm(Dc[0], 0, 0x1010); }   // x=-1 := x=0
            if (right_edge) { SR = __byte_perm(Sc[7], 0, 0x3232); DR = __byte_perm(Dc[7], 0, 0x3232); }  // x=W := x=W-1
            uint32_t So[9], Do[9];
            So[0] = __byte_perm(SL, Sc[0], 0x5432); Do[0] = __byte_perm(DL, Dc[0], 0x5432);
#pragma unroll
            for (int j = 1; j < 8; j++) {
                So[j] = __byte_perm(Sc[j - 1], Sc[j], 0x5432);
                Do[j] = __byte_perm(Dc[j - 1], Dc[j], 0x5432);
            }
            So[8] = __byte_perm(Sc[7], SR, 0x5432); Do[8] = __byte_perm(Dc[7], DR, 0x5432);
            uint32_t dx[8], dy[8], Mw[8], acc = 0;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                dx[j] = h2sub(So[j + 1], So[j]);
                dy[j] = h2fma2(Dc[j], h2add(Do[j], Do[j + 1]));
                Mw[j] = h2abs_sum(dx[j], dy[j]);
                const uint32_t gt = __hgt2_mask(*reinterpret_cast<const __half2 *>(&Mw[j]),
                                                *reinterpret_cast<const __half2 *>(&low2));      // 0xFFFF per half: M > low
                acc |= gt & ((1u << (2 * j)) | (1u << (2 * j + 17)));
            }
            cand_new = (acc | (acc >> 16)) & own_mask;
            uint4 *mrow = reinterpret_cast<uint4 *>(Mring + sc + xb);
            if (!row_ok) {                                       // warp-uniform, first / last row of the frame only
                cand_new = 0;
#pragma unroll
                for (int j = 0; j < 8; j++) Mw[j] = 0;
            }
            if (in_img) { mrow[0] = make_uint4(Mw[0], Mw[1], Mw[2], Mw[3]); mrow[1] = make_uint4(Mw[4], Mw[5], Mw[6], Mw[7]); }
            uint4 *xrow = reinterpret_cast<uint4 *>(DXr + (c & 1) * 512 + xb);
            xrow[0] = make_uint4(dx[0], dx[1], dx[2], dx[3]); xrow[1] = make_uint4(dx[4], dx[5], dx[6], dx[7]);
            uint4 *yrow = reinterpret_cast<uint4 *>(DYr + (c & 1) * 512 + xb);
            yrow[0] = make_uint4(dy[0], dy[1], dy[2], dy[3]); yrow[1] = make_uint4(dy[4], dy[5], dy[6], dy[7]);
        }
        __syncwarp();                                            // row c of the ring is visible to every lane
        if (c >= q0 + 1) {                                       // NMS of row n = c-1 (rows n-1, n, n+1 in slots sa, sb, sc)
            const int n = c - 1;
            const uint16_t *Ma = Mring + sa, *Mb = Mring + sb, *Mc = Mring + sc;
            const uint16_t *dxp = DXr + (n & 1) * 512, *dyp = DYr + (n & 1) * 512;
            uint32_t keep = 0, strong = 0, rem = cand_prev;
            while (rem) {
                const int p = __ffs(rem) - 1;
                rem &= rem - 1;
                const uint32_t x = xb + p;
                const int m = Mb[x];
                const uint32_t xr = dxp[x], yr = dyp[x];
                const int a = (int)(xr & 0x7FFFu), b = (int)(yr & 0x7FFFu);
                const int tg22x = a * 13573, ay = b << 15;
                const uint16_t *p1, *p2;
                int ge;                                          // second comparison is >= for the axis-aligned sectors
                if (ay < tg22x) { p1 = Mb + x - 1; p2 = Mb + x + 1; ge = 1; }                     // horizontal gradient
                else if (ay > tg22x + (a << 16)) { p1 = Ma + x; p2 = Mc + x; ge = 1; }              // vertical
                else {                                           // diagonal: along (+1,+1) when the signs agree
                    const int d = ((xr ^ yr) & 0x8000u) ? 1 : -1;
                    p1 = Ma + x + d; p2 = Mc + x - d; ge = 0;
                }
                const int n1 = *p1, n2 = *p2;
                if (m > n1 && m + ge > n2) {
                    keep |= 1u << p;
                    if (m > high) strong |= 1u << p;
                }
            }
            const uint32_t v = keep | (strong << 16);
            const uint32_t ov = __shfl_down_sync(0xffffffffu, v, 1);
            if (writer) {
                Cw[out_idx] = (v & 0xFFFFu) | (ov << 16);
                Sw[out_idx] = (v >> 16) | (ov & 0xFFFF0000u);
            }
            out_idx += WW;
        }
        __syncwarp();                                            // all reads of slot sa done before it is rewritten
        cand_prev = cand_new;
        const int t = sa; sa = sb; sb = sc; sc = t;
    };
    for (int c = q0 - 1;;) {
        step(std::integral_constant<int, 0>{}, c);
        if (++c > q1) break;
        step(std::integral_constant<int, 1>{}, c);
        if (++c > q1) break;
    }
}


// ---- K2a: Sobel + NMS + double threshold as a persistent warp-task kernel ---------------------------
// Warps pull (frame, band, strip) tasks from a global counter and write the candidate plane C and the
// strong plane S (32 px per word) to global memory; perfectly load-balanced, no barriers at all.
constexpr int K2A_WARPS = 4;
constexpr int K2A_CTAS = 6;             // CTAs per SM

__global__ void __launch_bounds__(K2A_WARPS * 32, K2A_CTAS) k2a_sobel_nms(const uint8_t *__restrict__ blur, const uint32_t *__restrict__ hist,
                                                               const uint8_t *__restrict__ lut_low,
                                                               const uint8_t *__restrict__ lut_high, int4 *__restrict__ thr,
                                                               uint32_t *__restrict__ c_bits, uint32_t *__restrict__ s_bits,
                                                               int *__restrict__ task_counter, int n_frames, int H, int W,
                                                               int band_rows, int tail_frames, int tail_rows)
{
    __shared__ __align__(16) uint16_t k2a_sm[K2A_WARPS][K2A_WSM];
    const int lane = threadIdx.x & 31;
    const int WW = (W + 31) / 32;
    const int n_strips = (W + STRIP_OUT - 1) / STRIP_OUT;
    // tasks in hand-out order: the first n_frames - tail_frames frames in bands of band_rows rows, the rest in thinner
    // bands so the end-of-kernel tail is short (same scheme as K1F)
    const int n_bands = (H + band_rows - 1) / band_rows, n_bands_t = (H + tail_rows - 1) / tail_rows;
    const int n_main = (n_frames - tail_frames) * n_bands * n_strips;
    const int n_tasks = n_main + tail_frames * n_bands_t * n_strips;
    for (;;) {
        int task = 0;
        if (lane == 0) task = atomicAdd(task_counter, 1);
        task = __shfl_sync(0xffffffffu, task, 0);
        if (task >= n_tasks) break;
        const bool tail = task >= n_main;
        const int tt = tail ? task - n_main : task, nb = tail ? n_bands_t : n_bands, br = tail ? tail_rows : band_rows;
        const int strip = tt % n_strips, band = (tt / n_strips) % nb;
        const int f = tt / (n_strips * nb) + (tail ? n_frames - tail_frames : 0);
        const int m2 = median_x2_warp(hist + f * 256, (long long)H * W, lane);
        int low = lut_low[m2], high = lut_high[m2];
        if (low > high) { int t = low; low = high; high = t; }
        if (band == 0 && strip == 0 && lane == 0) thr[f] = make_int4(m2, low, high, 0);
        const int q0 = band * br, q1 = min(q0 + br, H);
        canny_rows(H, W, WW, blur + (size_t)f * H * W, strip, q0, q1, c_bits + (size_t)f * H * WW,
                   s_bits + (size_t)f * H * WW, lane, low, high, k2a_sm[threadIdx.x >> 5]);
    }
}

// flood the seed bits of n along the runs of c (n subset of c) inside one 32-bit word
__device__ __forceinline__ uint32_t flood_word(uint32_t n, uint32_t c)
{
    uint32_t up = (((c + n) ^ c) & c) | n;
    uint32_t cr = __brev(c), ur = __brev(up);
    uint32_t dn = (((cr + ur) ^ cr) & cr) | ur;
    return __brev(dn);
}

// One hysteresis step on word (r, w) of the band: promote the weak pixels of the word that touch a strong pixel
// of the 3x3 word neighbourhood, then flood along the runs inside the word.  On a change the eight neighbouring
// words are flagged in the dirty map D, which is what later passes look at instead of re-checking every word.
__device__ __forceinline__ void mark_sides(volatile uint8_t *D, int Rv, int r, int w, int WW, uint32_t nb)
{
    // newly set bits reach a neighbouring word only from bit 0 / bit 31
    const int ra = max(r - 1, 0), rb = min(r + 1, Rv - 1);
    if ((nb & 1u) && w > 0)
        for (int q = ra; q <= rb; q++) D[q * WW + w - 1] = 1;
    if ((nb >> 31) && w < WW - 1)
        for (int q = ra; q <= rb; q++) D[q * WW + w + 1] = 1;
}

// returns the bits newly set in word (r, w); 0 = nothing changed
__device__ __forceinline__ uint32_t visit(const uint32_t *C, uint32_t *S, int r, int w, int WW)
{
    const uint32_t c = C[r * WW + w];
    uint32_t *sp = S + (r + 1) * WW + w;
    const uint32_t s = *sp;
    if ((c & ~s) == 0) return 0;
    const uint32_t v = sp[-WW] | s | sp[WW];
    uint32_t l = 0, rr = 0;
    if (w > 0) l = sp[-WW - 1] | sp[-1] | sp[WW - 1];
    if (w < WW - 1) rr = sp[-WW + 1] | sp[1] | sp[WW + 1];
    const uint32_t dil = v | (v << 1) | (v >> 1) | (l >> 31) | (rr << 31);
    uint32_t n = s | (c & dil);
    if (n == s) return 0;
    n = flood_word(n, c);
    atomicOr(sp, n);                    // result not awaited: bits somebody else set meanwhile only cause redundant flags
    return n & ~s;
}

__device__ __forceinline__ void mark_sides_cold(uint32_t dA, int Rv, int r, int w, int WW, uint32_t nb)
{
    // shared-memory byte address form of mark_sides (rare path of the column walk)
    const int ra = max(r - 1, 0), rb = min(r + 1, Rv - 1);
    const uint32_t one = 1;
    if ((nb & 1u) && w > 0)
        for (int q = ra; q <= rb; q++) asm volatile("st.shared.u8 [%0], %1;" ::"r"(dA + (q - r) * WW - 1), "r"(one) : "memory");
    if ((nb >> 31) && w < WW - 1)
        for (int q = ra; q <= rb; q++) asm volatile("st.shared.u8 [%0], %1;" ::"r"(dA + (q - r) * WW + 1), "r"(one) : "memory");
}

// Follow a promotion straight up or down its column word: only the pixels of the next row that touch the bits just
// set can change, so a step is two loads, a dilation and an in-word flood.  Everything the walk does not handle itself
// (the row behind it, the words to either side) is flagged dirty for the next pass.  Few threads walk while the rest
// of the CTA waits, so the loop is written for a short dependent-instruction chain: 32-bit shared addresses stepped
// by a constant, fire-and-forget atomic ORs (other walkers may be in the same word), the side flags out of the way.
__device__ __forceinline__ void chase_column(uint32_t cA, uint32_t sA, uint32_t dA, int Rv, int r, int w, int WW,
                                             uint32_t nb, int dir)
{
    const int wstep = dir * WW * 4, dstep = dir * WW;      // cA = &C[r][w], sA = &S[r+1][w], dA = &D[r][w]
    const uint32_t one = 1;
    for (;;) {
        r += dir;
        if ((unsigned)r >= (unsigned)Rv) return;
        cA += wstep; sA += wstep; dA += dstep;
        uint32_t c, sv;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(c) : "r"(cA));
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(sv) : "r"(sA));
        const uint32_t t = c & ~sv & (nb | (nb << 1) | (nb >> 1));
        if (!t) return;
        const uint32_t n = flood_word(sv | t, c);
        asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(sA), "r"(n) : "memory");
        nb = n & ~sv;
        asm volatile("st.shared.u8 [%0], %1;" ::"r"(dA - dstep), "r"(one) : "memory");   // the row behind
        if (nb & 0x80000001u) mark_sides_cold(dA, Rv, r, w, WW, nb);
    }
}

// ---- K2t: thresholds + candidate / strong planes from the fused edge kernel's output -----------------------------
// k1_fused leaves, per frame, the NMS survivors K (bit-plane) and their magnitudes V = min(m, 256) - 1 (byte plane, only
// survivors' bytes valid) plus the histogram.  Here the median and the two Canny thresholds are formed (np.median + the
// host LUT, lane_detector.py:79-81) and every survivor is classified: candidate iff m > low, strong iff m > high, i.e.
// V >= low / V >= high.  One thread per 32-px word, 32 bytes of V fetched only for words that have survivors; massively
// parallel, so the dependent V fetch costs nothing here (inside the hysteresis cluster it sat on the critical path).
// A frame whose true low is below the floor `pre` k1_fused used (the sampled estimate was too high) is flagged and
// listed for the redo pass instead.
struct K2tArgs {
    const uint32_t *k_bits;            // [n][H][WW]
    const uint8_t *v_plane;            // [n][H][W]
    int4 *thr;                         // [n] (median_x2, low, high, floor used), written by k1_fused
    const int *pre;                    // [n] floor k1_fused used for this pass
    const int *redo_flag;              // [n] first pass: frames listed for the redo pass are skipped
    const int *frame_list, *n_list;    // redo pass: frames to process (null = all)
    uint32_t *c_bits, *s_bits;         // [n][H][WW]
    int H, W, WW, words_per_cta;
};

__global__ void __launch_bounds__(256) k2t_threshold(K2tArgs A)
{
    // first pass: blockIdx.y = frame.  Redo pass: a few rows of CTAs walk the (normally empty) list of frames.
    const int n_list = A.frame_list ? *A.n_list : (int)gridDim.y;
    for (int fi = blockIdx.y; fi < n_list; fi += gridDim.y) {
        const int f = A.frame_list ? A.frame_list[fi] : fi;
        const int tid = threadIdx.x;
        // thresholds and the redo decision were formed by the warp of k1_fused that finished the frame last
        const int4 t = A.thr[f];
        if (!A.frame_list && A.redo_flag[f]) continue;          // this frame's planes are rebuilt in the redo pass
        if (A.frame_list && blockIdx.x == 0 && tid == 0) A.thr[f] = make_int4(t.x, t.y, t.z, A.pre[f]);
        const int s_low = t.y, s_high = t.z;
        const uint32_t lo4 = (uint32_t)s_low * 0x01010101u, hi4 = (uint32_t)s_high * 0x01010101u;
        const int n_words = A.H * A.WW;
        const uint32_t *kb = A.k_bits + (size_t)f * n_words;
        uint32_t *cb = A.c_bits + (size_t)f * n_words, *sb = A.s_bits + (size_t)f * n_words;
        const uint8_t *vb = A.v_plane + (size_t)f * A.H * A.W;
        auto ge_bits = [](const uint4 &a, const uint4 &b, uint32_t t4) {
            const uint32_t wds[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
            uint32_t m = 0;
#pragma unroll
            for (int q = 0; q < 8; q++)     // per byte 0/1 (V >= t), gathered into a nibble by one multiply
                m |= ((((__vcmpgeu4(wds[q], t4) & 0x01010101u) * 0x01020408u) >> 24) & 0xFu) << (4 * q);
            return m;
        };
        const int w0 = blockIdx.x * A.words_per_cta, w1 = min(w0 + A.words_per_cta, n_words);
        // eight words per thread, all K words requested before any is looked at
        uint32_t k[8];
#pragma unroll
        for (int u = 0; u < 8; u++) {
            const int i = w0 + tid + u * 256;
            k[u] = i < w1 ? __ldg(kb + i) : 0u;
        }
#pragma unroll
        for (int u = 0; u < 8; u++) {
            const int i = w0 + tid + u * 256;
            if (i >= w1) break;
            uint32_t cw = 0, sw = 0;
            if (k[u]) {
                const int r = i / A.WW, w = i - r * A.WW;
                const uint4 *vp = reinterpret_cast<const uint4 *>(vb + (size_t)r * A.W + w * 32);
                const uint4 a = __ldg(vp);
                const uint4 b = (w * 32 + 16 < A.W) ? __ldg(vp + 1) : make_uint4(0, 0, 0, 0);
                cw = k[u] & ge_bits(a, b, lo4);
                sw = k[u] & ge_bits(a, b, hi4);
            }
            cb[i] = cw;
            sb[i] = sw;
        }
    }
}

__global__ void __launch_bounds__(K2T, 3) k2_canny_cluster(K2Args A)
{
    extern __shared__ __align__(128) uint32_t smem[];
#ifdef LANE_K2_PROF
    int npass = 0; long long tps[8] = {0, 0, 0, 0, 0, 0, 0, 0}; long long tPm = 0; long long t0 = clock64(), tL = 0, tC0 = 0, tX = 0, tP3 = 0, tA = 0, tB = 0, tCc = 0, tD = 0, tmark = t0;
#define K2TICK(acc) do { long long n_ = clock64(); acc += n_ - tmark; tmark = n_; } while (0)
#else
#define K2TICK(acc) do { } while (0)
#endif
    cg::cluster_group cluster = cg::this_cluster();
    const int G = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
    int f = blockIdx.x / G;
    if (A.frame_list) {                          // redo pass: only the listed frames (the whole cluster leaves together)
        if (f >= *A.n_list) return;
        f = A.frame_list[f];
    }
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int H = A.H, WW = A.WW, R = A.R;
    if (A.skip_flag && !A.frame_list && A.skip_flag[f]) return;      // cluster-uniform: every CTA reads the same flag
    const int b0 = rank * R, b1 = min(b0 + R, H), Rv = max(b1 - b0, 0);
    uint32_t *C = smem;                         // [R][WW]
    uint32_t *S = smem + (size_t)R * WW;        // [R+2][WW], row 0 / Rv+1 = neighbour bands
    int *rowoff = reinterpret_cast<int *>(S + (size_t)(R + 2) * WW);   // [R+1]
    volatile uint8_t *D = reinterpret_cast<volatile uint8_t *>(rowoff + R + 1);          // [R][WW] dirty flags of the hysteresis passes
    __shared__ int s_flag, s_total, s_base, s_red[K2T / 32];
    __shared__ __align__(8) unsigned long long s_bar;

    // ---- phase 1 ran in k2a_sobel_nms: load this band's candidate / strong planes.  A band is one contiguous
    // run of Rv*WW words in each plane, so two bulk copies (TMA, completion on an mbarrier) bring it in.
    {
        const uint32_t *cg = A.c_bits + ((size_t)f * H + b0) * WW, *sg = A.s_bits + ((size_t)f * H + b0) * WW;
        const bool bulk = (WW % 4 == 0) && Rv > 0;
        if (bulk) {
            const uint32_t bar = smem_u32(&s_bar);
            if (tid == 0) {
                mbar_init(bar, 1);
                asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            }
            __syncthreads();
            if (tid == 0) {
                const uint32_t bytes = (uint32_t)Rv * WW * 4u;
                mbar_expect_tx(bar, 2 * bytes);
                bulk_g2s(smem_u32(C), cg, bytes, bar);
                bulk_g2s(smem_u32(S + WW), sg, bytes, bar);
            }
        } else {
            for (int i = tid; i < Rv * WW; i += K2T) { C[i] = cg[i]; S[WW + i] = sg[i]; }
        }
        for (int i = tid; i < WW; i += K2T) { S[i] = 0; S[(size_t)(Rv + 1) * WW + i] = 0; }
        for (int i = tid; i < (Rv * WW + 3) / 4; i += K2T) reinterpret_cast<volatile uint32_t *>(D)[i] = 0;
        if (bulk) mbar_wait(smem_u32(&s_bar), 0);
    }
    __syncthreads();
    K2TICK(tL);

    // ---- phase 2: hysteresis.  Work items are single 32-px words.  The first pass looks at every word of the band
    // (thread t takes words t, t+256, ... so the words of one column, where vertical chains sit, land on different
    // threads); a promotion is followed up and down its column at once, and flags the words beside it in the dirty
    // map.  Later passes only look at flagged words, until a pass changes nothing.  S only grows, all updates are
    // atomic ORs, and whoever sets a bit flags every word that bit can affect, so the fixed point is the closure.
    int rounds = 0;
    {
        uint32_t *S_up = rank > 0 ? cluster.map_shared_rank(S, rank - 1) : nullptr;
        uint32_t *S_dn = rank < G - 1 ? cluster.map_shared_rank(S, rank + 1) : nullptr;
        const int n_words = Rv * WW;
        auto visit_chase = [&](int i) {                   // i = r * WW + w
            const int r = i / WW, w = i - r * WW;
            const uint32_t nb = visit(C, S, r, w, WW);
            if (!nb) return false;
            mark_sides(D, Rv, r, w, WW, nb);
            const uint32_t cA = smem_u32(C + i), sA = smem_u32(S + WW + i);
            const uint32_t dA = smem_u32(const_cast<uint8_t *>(D) + i);
            chase_column(cA, sA, dA, Rv, r, w, WW, nb, +1);
            chase_column(cA, sA, dA, Rv, r, w, WW, nb, -1);
            return true;
        };
        K2TICK(tPm);
        auto converge = [&](bool full) {
            bool any_change = false;
            for (;;) {
#ifdef LANE_K2_PROF
                if (npass < 8) tps[npass] = clock64() - t0;
                npass++;
#endif
                bool ch = false;
                if (full) {
#pragma unroll 4
                    for (int i = tid; i < n_words; i += K2T)
                        if (C[i] & ~S[WW + i]) {
                            D[i] = 0;
                            ch |= visit_chase(i);
                        }
                } else {
                    const volatile uint32_t *D4 = reinterpret_cast<const volatile uint32_t *>(D);
                    for (int q = tid; q < (n_words + 3) / 4; q += K2T) {
                        uint32_t fl = D4[q];
                        while (fl) {                          // clear and visit exactly the flags that were seen set
                            const int k = (__ffs(fl) - 1) >> 3, i = 4 * q + k;
                            fl &= ~(0xFFu << (8 * k));
                            D[i] = 0;
                            if (i < n_words) ch |= visit_chase(i);
                        }
                    }
                }
                full = false;
                if (!__syncthreads_or(ch)) break;
                any_change = true;
            }
            return any_change;
        };
        converge(true);
        K2TICK(tC0);
        rounds = 1;
        // Bands then trade boundary rows.  A round ends the loop when NO band promoted anything after seeing its
        // neighbours' latest rows -- the usual case is one round (edges that cross a band boundary are strong on
        // both sides already), so the whole frame costs two cluster barriers.
        while (G > 1) {
            cluster.sync();                              // every band locally stable: boundary rows are final for this round
            for (int w = tid; w < WW; w += K2T) {
                if (S_up) S[w] = S_up[(size_t)R * WW + w];
                if (S_dn && Rv > 0) S[(size_t)(Rv + 1) * WW + w] = S_dn[WW + w];
                if (Rv > 0) { D[w] = 1; D[(Rv - 1) * WW + w] = 1; }     // only the boundary rows can react to the new halo rows
            }
            __syncthreads();
            const bool changed = converge(false);
            if (tid == 0) s_flag = changed;
            cluster.sync();
            int any = 0;
            if (tid < G) any = *cluster.map_shared_rank(&s_flag, tid);
            any = __syncthreads_or(any);
            if (!any) break;
            rounds++;
        }
    }

    K2TICK(tX);
    // ---- phase 3: outputs.  One fully parallel pass writes the edge plane, counts edges and forms the ROI-masked
    // plane in shared memory (the candidate plane is no longer needed, its storage is reused), so that the
    // row-major point list below never waits on global memory.
    const LaneGeom &g = A.g;
    const int y0 = max(b0, g.by0), y1 = min(b1, g.by1);
    const uint32_t *roi = A.roi_bits + (A.roi_index ? (size_t)A.roi_index[f] * A.roi_stride : 0);
    uint32_t *Mk = C;                                     // [Rv][WW] masked edges of this band
    int cnt = 0;
    uint32_t *eb = A.edge_bits + ((size_t)f * H + b0) * WW;
    uint32_t *pm = A.pmask_bits + (size_t)f * g.bh * WW;
    const bool bulk_out = (WW % 4 == 0) && Rv > 0;
    if (bulk_out) {
        // The band of the edge plane is the strong plane as it stands, one contiguous block: a single bulk store.
        // The ROI rows of the mask arrive by bulk copy into the (now free) candidate plane, are ANDed with the edges
        // in place and leave by a second bulk store; threads touch only shared memory.
        const int nroi = max(y1 - y0, 0);
        uint32_t *Mroi = Mk + (size_t)(y0 - b0) * WW;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // hysteresis stores -> async proxy
        __syncthreads();
        if (tid == 0) {
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                         ::"l"(eb), "r"(smem_u32(S + WW)), "r"((uint32_t)Rv * WW * 4u) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            if (nroi > 0) {
                const uint32_t bar = smem_u32(&s_bar);
                mbar_expect_tx(bar, (uint32_t)nroi * WW * 4u);
                bulk_g2s(smem_u32(Mroi), roi + (size_t)y0 * WW, (uint32_t)nroi * WW * 4u, bar);
            }
        }
        for (int i = tid; i < Rv * WW; i += K2T) cnt += __popc(S[WW + i]);
        if (nroi > 0) {
            mbar_wait(smem_u32(&s_bar), 1);                               // second use of the barrier: phase parity 1
            const uint32_t *Sroi = S + WW + (size_t)(y0 - b0) * WW;
            for (int i = tid; i < nroi * WW; i += K2T) Mroi[i] &= Sroi[i];
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncthreads();
            if (tid == 0) {
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                             ::"l"(pm + (size_t)(y0 - g.by0) * WW), "r"(smem_u32(Mroi)), "r"((uint32_t)nroi * WW * 4u) : "memory");
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
        }
        if (tid == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // S is reused below
    } else {
        const uint32_t *rb = roi + (size_t)b0 * WW;
        for (int i = tid; i < Rv * WW; i += K2T) {
            const int r = i / WW, y = b0 + r;
            const uint32_t sv = S[WW + i];
            eb[i] = sv;
            cnt += __popc(sv);
            uint32_t m = 0;
            if (y >= g.by0 && y < g.by1) {
                m = sv & rb[i];
                pm[(size_t)(y - g.by0) * WW + (i - r * WW)] = m;
            }
            Mk[i] = m;
        }
    }
    for (int o = 16; o; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (lane == 0) s_red[wid] = cnt;
    __syncthreads();
    if (tid == 0) {
        int t = 0;
        for (int i = 0; i < K2T / 32; i++) t += s_red[i];
        if (t) atomicAdd(&A.n_edges[f], t);
        if (rank == 0) A.rounds[f] = rounds;
    }
    K2TICK(tA);
    // a thread per ROI row: running count per word (kept in the strong plane's storage, which is free now) and the
    // row total; block scan of the totals; then every (row, word) writes its own points, all in parallel
    const int nrows = max(y1 - y0, 0);
    uint32_t *Pfx = S + WW;                               // [Rv][WW] points of the row before word w
    for (int i = tid; i < nrows; i += K2T) {
        const uint32_t *row = Mk + (size_t)(y0 + i - b0) * WW;
        uint32_t *pf = Pfx + (size_t)(y0 + i - b0) * WW;
        int c = 0;
#pragma unroll 4
        for (int w = 0; w < WW; w++) { pf[w] = c; c += __popc(row[w]); }
        rowoff[y0 + i - b0] = c;
    }
    __syncthreads();
    if (wid == 0) {                                       // exclusive scan of the row counts
        int run = 0;
        for (int base = y0; base < y1; base += 32) {
            const int y = base + lane;
            const int v = y < y1 ? rowoff[y - b0] : 0;
            int inc = v;
            for (int o = 1; o < 32; o <<= 1) {
                int t = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o) inc += t;
            }
            if (y < y1) rowoff[y - b0] = run + inc - v;
            run += __shfl_sync(0xffffffffu, inc, 31);
        }
        if (lane == 0) s_total = run;
    }
    __syncthreads();
    K2TICK(tB);
    if (G > 1) cluster.sync();
    K2TICK(tCc);
    if (tid == 0) {
        int base = 0;
        for (int r = 0; r < rank; r++) base += *cluster.map_shared_rank(&s_total, r);
        s_base = base;
        if (s_total) atomicAdd(&A.n_points[f], s_total);
    }
    __syncthreads();
    uint32_t *out = A.points + (size_t)f * g.max_points + s_base;
    {
        const int cols = min(WW, K2T), rstep = max(1, K2T / WW);
        const int w0 = tid % cols, r0 = tid / cols;
        if (r0 < rstep)
            for (int w = w0; w < WW; w += cols)
                for (int i = r0; i < nrows; i += rstep) {
                    const int lr = y0 + i - b0;
                    uint32_t m = Mk[(size_t)lr * WW + w];
                    if (!m) continue;
                    int p = rowoff[lr] + (int)Pfx[(size_t)lr * WW + w];
                    const uint32_t hi = ((uint32_t)(y0 + i) << 16) | (uint32_t)(w * 32);
                    while (m) {
                        out[p++] = hi | (uint32_t)(__ffs(m) - 1);
                        m &= m - 1;
                    }
                }
    }
    K2TICK(tD);
    if (G > 1) cluster.sync();                            // keep s_total alive until every band has read it
    if (tid == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
#ifdef LANE_K2_PROF
    K2TICK(tP3);
    if (tid == 0 && f == 128) printf("k2b rank=%d total=%lld load=%lld pmask=%lld passes=%d [%lld %lld %lld %lld %lld %lld] converge0=%lld rounds(%d)=%lld p3: write=%lld counts=%lld csync=%lld points=%lld final=%lld\n", rank, clock64() - t0, tL, tPm, npass, tps[0], tps[1], tps[2], tps[3], tps[4], tps[5], tC0, rounds, tX, tA, tB, tCc, tD, tP3);
#endif
}

// byte map -> bit-plane (generic-width fallback path)
__global__ void k_bytes_to_bits(const uint8_t *__restrict__ bytes, uint32_t *__restrict__ bits, int rows, int W,
                                int row_stride, int WW)
{
    const int y = blockIdx.y, f = blockIdx.z;
    const uint8_t *src = bytes + ((size_t)f * rows + y) * row_stride;
    uint32_t *dst = bits + ((size_t)f * rows + y) * WW;
    for (int w = blockIdx.x * blockDim.x + threadIdx.x; w < WW; w += gridDim.x * blockDim.x) {
        uint32_t m = 0;
        for (int b = 0; b < 32; b++) {
            const int x = w * 32 + b;
            if (x < W && src[x]) m |= 1u << b;
        }
        dst[w] = m;
    }
}

// pmask[f][y-by0][w] = edge_bits[f][y][w] & roi_bits[roi_index[f]][y][w]  (generic-width fallback path)
__global__ void k_mask_rows(const uint32_t *__restrict__ edge_bits, const uint32_t *__restrict__ roi_bits,
                            const int *__restrict__ roi_index, size_t roi_stride, uint32_t *__restrict__ pmask_bits, int H,
                            int WW, int by0, int bh)
{
    const int f = blockIdx.y;
    if (roi_index) roi_bits += (size_t)roi_index[f] * roi_stride;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < bh * WW; i += gridDim.x * blockDim.x) {
        const int y = by0 + i / WW, w = i % WW;
        pmask_bits[(size_t)f * bh * WW + i] = edge_bits[((size_t)f * H + y) * WW + w] & roi_bits[(size_t)y * WW + w];
    }
}

}  // namespace

// Cluster geometry of K2b for a frame size: G CTAs per frame, R rows per band, dynamic shared memory; false when the
// frame does not fit (caller falls back to the generic byte-map kernels).
static bool k2b_plan(int H, int W, int *G_out, int *R_out, size_t *smem_out)
{
    const int WW = (W + 31) / 32;
    int G = 1;
    while (G < 16 && H > 160 * G) G *= 2;                // bands of up to 160 rows
    size_t smem = 0;
    int R = 0;
    for (;; G *= 2) {
        R = (H + G - 1) / G;
        smem = sizeof(uint32_t) * ((size_t)R * WW + (size_t)(R + 2) * WW) + sizeof(int) * (R + 1) + ((size_t)R * WW + 4);
        if (smem <= 200 * 1024 || G >= 16) break;
    }
    if (smem > 220 * 1024) return false;
    static bool configured[LANE_MAX_DEVICES];
    if (!configured[lane_cur_device()]) {
        cudaFuncSetAttribute(k2_canny_cluster, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
        cudaFuncSetAttribute(k2_canny_cluster, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
        configured[lane_cur_device()] = true;
    }
    *G_out = G; *R_out = R; *smem_out = smem;
    return true;
}

static cudaError_t k2b_launch(const K2Args &A, int G, size_t smem, int n, cudaStream_t st)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(n * G);
    cfg.blockDim = dim3(K2T);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = G; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, k2_canny_cluster, A);
}

// Unfused form: K2a (Sobel + NMS + thresholds from the blurred plane) then K2b.  Returns false when this frame geometry
// cannot take the cluster path (caller falls back to the generic byte-map kernels).
bool launch_canny_cluster(const uint8_t *blur, const uint32_t *hist, const uint8_t *lut_low, const uint8_t *lut_high,
                          const uint32_t *roi_bits, const int *roi_index, size_t roi_stride, int4 *thr, int *n_edges, int *rounds, uint32_t *points,
                          int *n_points, uint32_t *pmask_bits, uint32_t *edge_bits, uint32_t *c_bits, uint32_t *s_bits,
                          int *task_counter, LaneGeom g, int n, cudaStream_t st, int *launches)
{
    const int H = g.H, W = g.W, WW = (W + 31) / 32;
    if (W % 16 != 0 || ((uintptr_t)blur % 16) != 0) return false;
    int G = 1, R = 0;
    size_t smem = 0;
    if (!k2b_plan(H, W, &G, &R, &smem)) return false;
    const int sms = lane_sm_count();
    cudaMemsetAsync(task_counter, 0, sizeof(int), st);
    {
        const int n_strips = (W + STRIP_OUT - 1) / STRIP_OUT, warps = sms * K2A_CTAS * K2A_WARPS;
        // small batches: at least two tasks per resident warp, bands no thinner than 12 rows
        const long rows_per_warp = ((long)n * H * n_strips + 2 * warps - 1) / (2 * warps);
        const int band_rows = (int)std::max(12L, std::min(64L, rows_per_warp));
        int tail_frames = n >= 16 ? n / 16 : 0;
        const int tail_rows = std::max(12, band_rows / 3);
        if (tail_rows >= band_rows) tail_frames = 0;
        k2a_sobel_nms<<<sms * K2A_CTAS, K2A_WARPS * 32, 0, st>>>(blur, hist, lut_low, lut_high, thr, c_bits, s_bits, task_counter,
                                                                  n, H, W, band_rows, tail_frames, tail_rows);
    }
    K2Args A{};
    A.c_bits = c_bits; A.s_bits = s_bits; A.roi_bits = roi_bits; A.roi_index = roi_index; A.roi_stride = roi_stride;
    A.n_edges = n_edges; A.rounds = rounds; A.n_points = n_points; A.points = points;
    A.pmask_bits = pmask_bits; A.edge_bits = edge_bits;
    A.H = H; A.W = W; A.WW = WW; A.R = R; A.g = g;
    cudaMemsetAsync(n_edges, 0, sizeof(int) * n, st);
    cudaMemsetAsync(n_points, 0, sizeof(int) * n, st);
    cudaError_t e = k2b_launch(A, G, smem, n, st);
    if (e != cudaSuccess) { cudaGetLastError(); return false; }
    *launches += 2;
    return true;
}

// Fused form: thresholds + candidate / strong planes from k1_fused's K / V planes (k2t_threshold), then K2b.
// frame_list == null: first pass over frames 0..n-1; frames whose magnitude floor turned out to be above their true low
// are flagged, listed in redo_list and skipped.  frame_list == redo_list: the redo pass, after launch_fused_edge_redo
// has rebuilt those frames' planes with the exact floor.
bool launch_canny_cluster_fused(const uint32_t *k_bits, const uint8_t *v_plane, const uint32_t *hist, const uint8_t *lut_low,
                                const uint8_t *lut_high, const uint32_t *roi_bits, const int *roi_index, size_t roi_stride,
                                int4 *thr, const int *pre, int *pre_redo, int *redo_list, int *redo_count, int *redo_flag,
                                const int *frame_list, int *n_edges, int *rounds, uint32_t *points, int *n_points,
                                uint32_t *pmask_bits, uint32_t *edge_bits, uint32_t *c_bits, uint32_t *s_bits, LaneGeom g, int n,
                                cudaStream_t st, int *launches)
{
    const int H = g.H, W = g.W, WW = (W + 31) / 32;
    int G = 1, R = 0;
    size_t smem = 0;
    if (!k2b_plan(H, W, &G, &R, &smem)) return false;
    if (!frame_list) {
        cudaMemsetAsync(n_edges, 0, sizeof(int) * n, st);
        cudaMemsetAsync(n_points, 0, sizeof(int) * n, st);
    }
    K2tArgs T{};
    T.k_bits = k_bits; T.v_plane = v_plane; T.thr = thr; T.pre = frame_list ? pre_redo : pre;
    T.redo_flag = redo_flag; T.frame_list = frame_list; T.n_list = frame_list ? redo_count : nullptr;
    T.c_bits = c_bits; T.s_bits = s_bits; T.H = H; T.W = W; T.WW = WW;
    T.words_per_cta = 256 * 8;              // the kernel handles exactly eight words per thread
    dim3 tgrid((H * WW + T.words_per_cta - 1) / T.words_per_cta, frame_list ? std::min(n, 8) : n);
    k2t_threshold<<<tgrid, 256, 0, st>>>(T);
    K2Args A{};
    A.c_bits = c_bits; A.s_bits = s_bits; A.skip_flag = redo_flag;
    A.frame_list = frame_list; A.n_list = frame_list ? redo_count : nullptr;
    A.roi_bits = roi_bits; A.roi_index = roi_index; A.roi_stride = roi_stride;
    A.n_edges = n_edges; A.rounds = rounds; A.n_points = n_points; A.points = points;
    A.pmask_bits = pmask_bits; A.edge_bits = edge_bits;
    A.H = H; A.W = W; A.WW = WW; A.R = R; A.g = g;
    cudaError_t e = k2b_launch(A, G, smem, n, st);
    if (e != cudaSuccess) { cudaGetLastError(); return false; }
    *launches += 2;
    return true;
}

// edge pixels inside [x0,x1) x [y0,y1) of every frame's edge bit-plane (SceneClassifier's centre-region edge density,
// src/tagging/scene_classifier.py:148-150): one CTA per frame, popcounts of the masked words
namespace {
__global__ void __launch_bounds__(256) k_edge_count_rect(const uint32_t *__restrict__ edge_bits, int *__restrict__ counts, int H,
                                                         int WW, int x0, int y0, int x1, int y1)
{
    __shared__ int s_red[8];
    const int f = blockIdx.x, tid = threadIdx.x;
    const uint32_t *eb = edge_bits + (size_t)f * H * WW;
    const int w0 = x0 >> 5, w1 = (x1 + 31) >> 5, nw = w1 - w0;
    int cnt = 0;
    for (int i = tid; i < (y1 - y0) * nw; i += 256) {
        const int y = y0 + i / nw, w = w0 + i % nw;
        uint32_t m = eb[(size_t)y * WW + w];
        if (w == w0) m &= 0xFFFFFFFFu << (x0 & 31);
        if (w == w1 - 1 && (x1 & 31)) m &= 0xFFFFFFFFu >> (32 - (x1 & 31));
        cnt += __popc(m);
    }
    for (int o = 16; o; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((tid & 31) == 0) s_red[tid >> 5] = cnt;
    __syncthreads();
    if (tid == 0) {
        int t = 0;
        for (int i = 0; i < 8; i++) t += s_red[i];
        counts[f] = t;
    }
}
}  // namespace

void launch_edge_count_rect(const uint32_t *edge_bits, int *counts, int n, int H, int W, int x0, int y0, int x1, int y1,
                            cudaStream_t st)
{
    k_edge_count_rect<<<n, 256, 0, st>>>(edge_bits, counts, H, (W + 31) / 32, x0, y0, x1, y1);
}

void launch_bytes_to_bits(const uint8_t *bytes, uint32_t *bits, int n, int rows, int W, int row_stride,
                          cudaStream_t st, int *launches)
{
    const int WW = (W + 31) / 32;
    dim3 grid((WW + 63) / 64, rows, n);
    k_bytes_to_bits<<<grid, 64, 0, st>>>(bytes, bits, rows, W, row_stride, WW);
    if (launches) *launches += 1;
}

void launch_mask_rows(const uint32_t *edge_bits, const uint32_t *roi_bits, const int *roi_index, size_t roi_stride,
                      uint32_t *pmask_bits, LaneGeom g, int n, cudaStream_t st, int *launches)
{
    const int WW = (g.W + 31) / 32;
    if (g.bh <= 0) return;
    dim3 grid((g.bh * WW + 255) / 256, n);
    k_mask_rows<<<grid, 256, 0, st>>>(edge_bits, roi_bits, roi_index, roi_stride, pmask_bits, g.H, WW, g.by0, g.bh);
    if (launches) *launches += 1;
}
