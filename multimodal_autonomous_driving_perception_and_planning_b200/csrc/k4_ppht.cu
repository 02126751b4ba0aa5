// K4: exact progressive probabilistic Hough (cv2.HoughLinesP, lane_detector.py:94-101).
//
// The algorithm is sequential and randomised with a fixed seed (SURVEY.md A.6): points are drawn
// from the row-major list with the MWC generator RNG(0xFFFFFFFFFFFFFFFF), each votes 180 bins
// (float32 rho = x*cos + y*sin, separate multiply/add, round-half-even), and the first bin to reach
// the threshold triggers a fixed-point line walk that removes (and, for a good line, un-votes) the
// pixels on it.  Every angle is voted by exactly one thread, in point order, so it sees exactly the
// sequential vote counts; points are drawn in batches (the draw order never depends on the
// accumulator or the mask) and voted speculatively: the first triggering point of a batch is exact,
// later votes of the batch are rolled back and replayed after the walk.  Two kernels:
//   k4_ppht_v3  a cluster of CTAs per frame, accumulator in distributed shared memory (default)
//   k4_ppht_v2  one CTA per frame, accumulator in global memory (frames and ROIs v3 cannot take)
#include "lane_common.cuh"

#include <math.h>
#include <type_traits>
#include <stdio.h>
#include <stdlib.h>

__constant__ float c_ppht_cos[LANE_NUM_ANGLES], c_ppht_sin[LANE_NUM_ANGLES];

void lane_upload_tables()
{
    float pc[LANE_NUM_ANGLES], ps[LANE_NUM_ANGLES];
    const float theta = (float)(M_PI / 180.0);
    for (int n = 0; n < LANE_NUM_ANGLES; n++) {
        // HoughLinesP: cos/sin of double(n)*double(theta_f), narrowed to float (A.6)
        pc[n] = (float)cos((double)n * theta);
        ps[n] = (float)sin((double)n * theta);
    }
    cudaMemcpyToSymbol(c_ppht_cos, pc, sizeof(pc));
    cudaMemcpyToSymbol(c_ppht_sin, ps, sizeof(ps));
    lane_upload_tables_std();
}

namespace {

constexpr int LIST_CAP = 8192;    // point list kept in shared memory when it fits
constexpr unsigned SKIP = 0xFFFFFFFFu;

__device__ __forceinline__ int rho_of(int x, int y, float cs, float sn)
{
    // two float32 products, one float32 add, no FMA contraction, round half to even
    return __float2int_rn(__fadd_rn(__fmul_rn((float)x, cs), __fmul_rn((float)y, sn)));
}

__device__ __forceinline__ int rho_f(float x, float y, float cs, float sn)
{
    return __float2int_rn(__fadd_rn(__fmul_rn(x, cs), __fmul_rn(y, sn)));
}

struct WalkSetup {
    int x0, y0, dx0, dy0, xflag;
};

__device__ __forceinline__ void step_pixel(const WalkSetup &w, int k, int s, int &j1, int &i1)
{
    int dx = k ? -w.dx0 : w.dx0, dy = k ? -w.dy0 : w.dy0;
    int x = w.x0 + s * dx, y = w.y0 + s * dy;
    if (w.xflag) { j1 = x; i1 = y >> 16; } else { j1 = x >> 16; i1 = y; }
}

// ---------------------------------------------------------------------------------------------
// v2: one CTA per frame; voter thread n < 180 owns angle n and its accumulator row.
//   * a producer warp draws the points (RNG + swap-remove on the shared-memory list) one batch
//     ahead of the six voter warps (double-buffered batches, one CTA barrier per batch);
//   * votes are issued eight deep before any result is inspected, so the L2 round trips overlap;
//   * accumulator cells are biased 16-bit counters packed two per word, and every angle only owns
//     the rho window the ROI can reach (host-computed from the mask's row spans with the same
//     float32 arithmetic), so a 1080p frame needs ~0.45 MB instead of the 4.3 MB of int32 cells over
//     the full rho range, and stays in L2.
constexpr int NV = 192;            // voter threads (180 active)
constexpr int NT2 = NV + 32;       // + producer warp
constexpr int BATCH2 = 64;
constexpr unsigned BIAS = 0x4040u; // cudaMemset(0x40) per byte

__device__ __forceinline__ void bar_voters() { asm volatile("bar.sync 1, %0;" ::"n"(NV) : "memory"); }

__device__ __forceinline__ int cell_add(uint32_t *acc32, int cell, int delta)   // returns the value BEFORE the add
{
    const unsigned sh = (cell & 1) * 16;
    const unsigned old = atomicAdd(&acc32[cell >> 1], (unsigned)delta << sh);
    return (int)((old >> sh) & 0xFFFFu) - (int)BIAS;
}
__device__ __forceinline__ void cell_red(uint32_t *acc32, int cell, int delta)
{
    atomicAdd(&acc32[cell >> 1], (unsigned)delta << ((cell & 1) * 16));
}

__global__ void __launch_bounds__(NT2) k4_ppht_v2(uint32_t *__restrict__ points_all, const int *__restrict__ n_points,
                                                  uint32_t *__restrict__ pmask_all, uint32_t *__restrict__ accum_all,
                                                  const int2 *__restrict__ win, int cells_per_frame,
                                                  int32_t *__restrict__ lines_all, int *__restrict__ n_lines,
                                                  LaneGeom g, LaneHoughParams hp, int only_flagged)
{
    __shared__ uint32_t s_list[LIST_CAP];
    __shared__ uint32_t s_buf[2][BATCH2];
    if (only_flagged) {                             // clean-up pass behind v3: frames it could not take (n_lines == -1)
        if (n_lines[blockIdx.x] != -1) return;
        uint32_t *a = accum_all + (size_t)blockIdx.x * (cells_per_frame / 2);
        for (int i = threadIdx.x; i < cells_per_frame / 2; i += NT2) a[i] = BIAS | (BIAS << 16);
        __threadfence_block();
    }
    __shared__ int s_trig;
    __shared__ int s_redv[NV / 32], s_redn[NV / 32];
    __shared__ int s_end[2][2];
    __shared__ int s_nsteps[2];
    __shared__ int s_good;
    __shared__ uint32_t s_hits[NV];
    __shared__ int s_nhits;
    __shared__ WalkSetup s_walk;

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, f = blockIdx.x;
    const bool producer = wid == NV / 32;
    const bool active = tid < LANE_NUM_ANGLES;
    const int WW = (g.W + 31) / 32;
    uint32_t *pm = pmask_all + (size_t)f * g.bh * WW;
    int32_t *lines = lines_all + (size_t)f * g.max_segments * 4;
    uint32_t *acc32 = accum_all + (size_t)f * (cells_per_frame / 2);
    const float cs = active ? c_ppht_cos[tid] : 0.f, sn = active ? c_ppht_sin[tid] : 0.f;
    const int2 wn = active ? win[tid] : make_int2(0, 0);
    const int cell0 = wn.y - wn.x;                  // cell(r) = cell0 + r

    const int count0 = n_points[f];
    uint32_t *list = points_all + (size_t)f * g.max_points;
    if (count0 <= LIST_CAP) {
        for (int i = tid; i < count0; i += NT2) s_list[i] = list[i];
        list = s_list;
    }
    const int n_batches = (count0 + BATCH2 - 1) / BATCH2;
    uint64_t rng = 0xFFFFFFFFFFFFFFFFull;           // producer lane 0 only
    int remaining = count0;                         // producer lane 0 only
    int nl = 0;                                     // thread 0 only
    __syncthreads();

    auto draw = [&](uint32_t *buf) {                // producer lane 0: next min(BATCH2, remaining) points, in order
        const int P = remaining < BATCH2 ? remaining : BATCH2;
        for (int k = 0; k < P; k++) {
            rng = (uint64_t)(uint32_t)rng * 4164903690ull + (uint32_t)(rng >> 32);
            const int idx = (int)((uint32_t)rng % (uint32_t)remaining);
            buf[k] = list[idx];
            list[idx] = list[remaining - 1];
            remaining--;
        }
    };
    if (producer && lane == 0 && n_batches > 0) draw(s_buf[0]);
    __syncthreads();

    for (int bi = 0; bi < n_batches; bi++) {
        uint32_t *batch = s_buf[bi & 1];
        const int P = min(BATCH2, count0 - bi * BATCH2);
        if (producer) {
            if (lane == 0 && bi + 1 < n_batches) draw(s_buf[(bi + 1) & 1]);
        } else {
            int k0 = 0;
            while (k0 < P) {
                if (tid == 0) s_trig = BATCH2;
                if (tid >= k0 && tid < P) {              // drop points an earlier walk already removed
                    const uint32_t pt = batch[tid];
                    if (pt != SKIP) {
                        const int x = pt & 0xFFFF, y = pt >> 16;
                        if (!((__ldcg(&pm[(y - g.by0) * WW + (x >> 5)]) >> (x & 31)) & 1u)) batch[tid] = SKIP;
                    }
                }
                bar_voters();
                if (active) {                            // thread n votes its own row, in order, eight deep
                    int first = BATCH2;
                    for (int kk = k0; kk < P; kk += 8) {
                        int v[8];
#pragma unroll
                        for (int u = 0; u < 8; u++) {
                            const int k = kk + u;
                            const uint32_t pt = k < P ? batch[k] : SKIP;
                            v[u] = -0x40000000;
                            if (pt != SKIP) v[u] = cell_add(acc32, cell0 + rho_of(pt & 0xFFFF, pt >> 16, cs, sn), 1);
                        }
#pragma unroll
                        for (int u = 0; u < 8; u++)
                            if (v[u] + 1 >= hp.threshold) first = min(first, kk + u);
                    }
                    if (first < BATCH2) atomicMin(&s_trig, first);
                }
                bar_voters();
                const int t = s_trig;
                if (t == BATCH2) break;
                if (active) {                            // roll back the speculative votes behind the trigger
                    for (int k = t + 1; k < P; k++) {
                        const uint32_t pt = batch[k];
                        if (pt != SKIP) cell_red(acc32, cell0 + rho_of(pt & 0xFFFF, pt >> 16, cs, sn), -1);
                    }
                }
                const uint32_t tp = batch[t];
                const int px = tp & 0xFFFF, py = tp >> 16;
                int bv = -2147483647, bn = 0x7fffffff;
                if (active) { bv = cell_add(acc32, cell0 + rho_of(px, py, cs, sn), 0); bn = tid; }
                for (int o = 16; o; o >>= 1) {
                    int ov = __shfl_xor_sync(0xffffffffu, bv, o), on = __shfl_xor_sync(0xffffffffu, bn, o);
                    if (ov > bv || (ov == bv && on < bn)) { bv = ov; bn = on; }
                }
                if (lane == 0) { s_redv[wid] = bv; s_redn[wid] = bn; }
                bar_voters();
                if (tid == 0) {
                    int mv = s_redv[0], mn = s_redn[0];
                    for (int w = 1; w < NV / 32; w++)
                        if (s_redv[w] > mv || (s_redv[w] == mv && s_redn[w] < mn)) { mv = s_redv[w]; mn = s_redn[w]; }
                    float a = -c_ppht_sin[mn], b = c_ppht_cos[mn];
                    WalkSetup w;
                    w.x0 = px; w.y0 = py;
                    if (fabsf(a) > fabsf(b)) {
                        w.xflag = 1;
                        w.dx0 = a > 0 ? 1 : -1;
                        w.dy0 = __float2int_rn(__fdiv_rn(__fmul_rn(b, 65536.0f), fabsf(a)));
                        w.y0 = (py << 16) + 32768;
                    } else {
                        w.xflag = 0;
                        w.dy0 = b > 0 ? 1 : -1;
                        w.dx0 = __float2int_rn(__fdiv_rn(__fmul_rn(a, 65536.0f), fabsf(b)));
                        w.x0 = (px << 16) + 32768;
                    }
                    s_walk = w;
                }
                bar_voters();
                const WalkSetup w = s_walk;
                if (wid < 2) {                           // pass 1: one warp per direction, 32 steps per ballot
                    const int k = wid;
                    int last = 0;
                    bool done = false;
                    for (int base = 0; !done; base += 32) {
                        int j1, i1;
                        step_pixel(w, k, base + lane, j1, i1);
                        bool ib = j1 >= 0 && j1 < g.W && i1 >= 0 && i1 < g.H;
                        bool hit = false;
                        if (ib && i1 >= g.by0 && i1 < g.by1)
                            hit = ((__ldcg(&pm[(i1 - g.by0) * WW + (j1 >> 5)]) >> (j1 & 31)) & 1u) != 0;
                        unsigned IB = __ballot_sync(0xffffffffu, ib), Hh = __ballot_sync(0xffffffffu, hit);
                        int limit = (~IB) ? __ffs(~IB) - 1 : 32;
                        if (limit < 32) Hh &= (1u << limit) - 1u;
                        while (Hh) {
                            int p = base + __ffs(Hh) - 1;
                            if (p - last > hp.max_gap + 1) { done = true; break; }
                            last = p;
                            Hh &= Hh - 1;
                        }
                        if (!done) {
                            if (limit < 32) done = true;
                            else if (base + 31 - last > hp.max_gap) done = true;
                        }
                    }
                    if (lane == 0) {
                        int j1, i1;
                        step_pixel(w, k, last, j1, i1);
                        s_end[k][0] = j1; s_end[k][1] = i1;
                        s_nsteps[k] = last + 1;
                    }
                }
                bar_voters();
                if (tid == 0) {
                    int good = abs(s_end[1][0] - s_end[0][0]) >= hp.min_len || abs(s_end[1][1] - s_end[0][1]) >= hp.min_len;
                    s_good = good;
                    if (good) {
                        if (nl < g.max_segments) {
                            lines[4 * nl + 0] = s_end[0][0]; lines[4 * nl + 1] = s_end[0][1];
                            lines[4 * nl + 2] = s_end[1][0]; lines[4 * nl + 3] = s_end[1][1];
                        }
                        nl++;
                    }
                }
                for (int k = 0; k < 2; k++) {            // pass 2: clear the segment's pixels, un-vote them if good
                    const int ns = s_nsteps[k];
                    for (int base = 0; base < ns; base += NV) {
                        if (tid == 0) s_nhits = 0;
                        bar_voters();
                        int s = base + tid;
                        if (s < ns) {
                            int j1, i1;
                            step_pixel(w, k, s, j1, i1);
                            if (i1 >= g.by0 && i1 < g.by1 && j1 >= 0 && j1 < g.W) {
                                const uint32_t bit = 1u << (j1 & 31);
                                if (atomicAnd(&pm[(i1 - g.by0) * WW + (j1 >> 5)], ~bit) & bit)
                                    s_hits[atomicAdd(&s_nhits, 1)] = ((uint32_t)i1 << 16) | (uint32_t)j1;
                            }
                        }
                        bar_voters();
                        if (s_good && active) {
                            const int nh = s_nhits;
                            for (int h = 0; h < nh; h++) {
                                const uint32_t pt = s_hits[h];
                                cell_red(acc32, cell0 + rho_of(pt & 0xFFFF, pt >> 16, cs, sn), -1);
                            }
                        }
                        bar_voters();
                    }
                }
                k0 = t + 1;
            }
        }
        __syncthreads();
    }
    if (tid == 0) n_lines[f] = nl;
}


// ---------------------------------------------------------------------------------------------
// v3: accumulator in (distributed) shared memory.  Global atomics bound v2 (85 M votes per 256
// frames against the L2 atomic rate), so here a cluster of G CTAs owns one frame and CTA r keeps
// the 16-bit cells of the angles n = r (mod G) in its own shared memory; each angle is still voted
// by exactly one thread, in point order, with plain shared-memory read-modify-writes (exact
// sequential counts, no atomics).  Every CTA draws the same point sequence (producer warp) and
// walks the same lines on its private copy of the mask, so the only traffic between CTAs is one
// 64-bit word per CTA per batch (first triggering point) and one per trigger (arg-max), exchanged
// through DSMEM slots with a sequence number -- no cluster barrier on the hot path.
constexpr int BATCH3 = 64;
constexpr int LIST_CAP3 = 3072;      // points of a frame kept in shared memory (the plan may settle for less to fit a smaller cluster)
constexpr int OVER_CAP3 = 131072;    // most points a frame may keep in the private global (L2) extension of its list

struct XchgSlots {
    unsigned long long v[2][16];   // [seq parity][source rank] = seq << 32 | payload
};

__device__ __forceinline__ uint32_t dsmem_addr(const void *local_smem_ptr, unsigned rank)
{
    uint32_t a = (uint32_t)__cvta_generic_to_shared(local_smem_ptr), r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(rank));
    return r;
}
// payload and sequence number travel in one 64-bit word, so relaxed accesses suffice (no fence, no L1 flush)
__device__ __forceinline__ void dsmem_store_release(uint32_t addr, unsigned long long v)
{
    asm volatile("st.relaxed.cluster.shared::cluster.b64 [%0], %1;" ::"r"(addr), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long smem_load_acquire(const unsigned long long *p)
{
    unsigned long long v;
    uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
    asm volatile("ld.relaxed.cluster.shared::cta.b64 %0, [%1];" : "=l"(v) : "r"(a) : "memory");
    return v;
}

// all-gather of one 32-bit payload per CTA; called by one thread per CTA.  op: 0 = min, 1 = max.
__device__ __forceinline__ uint32_t cluster_reduce(XchgSlots *slots, unsigned &seq, int G, int rank, uint32_t payload,
                                                   int op)
{
    seq++;
    const unsigned par = seq & 1;
    const unsigned long long word = ((unsigned long long)seq << 32) | payload;
    for (int p = 0; p < G; p++) dsmem_store_release(dsmem_addr(&slots->v[par][rank], p), word);
    uint32_t res = payload;
    for (int p = 0; p < G; p++) {
        unsigned long long w;
        do { w = smem_load_acquire(&slots->v[par][p]); } while ((unsigned)(w >> 32) != seq);
        const uint32_t q = (uint32_t)w;
        res = op ? max(res, q) : min(res, q);
    }
    return res;
}

constexpr int FLAG_CAP = 48;
constexpr unsigned CBIAS = 0x4000u;
constexpr int HITS_CAP = 512;        // cleared pixels of one un-vote round, packed (y << 16) | x
constexpr int WPT = 4;             // pass-1 walk steps per thread per round

__device__ __forceinline__ int scell_add(uint32_t *cells32, int cell, int delta)   // value BEFORE the add
{
    const unsigned sh = (cell & 1) * 16;
    const unsigned old = atomicAdd(&cells32[cell >> 1], (unsigned)delta << sh);
    return (int)((old >> sh) & 0xFFFFu) - (int)CBIAS;
}
__device__ __forceinline__ int scell_get(const uint32_t *cells32, int cell)
{
    return (int)((cells32[cell >> 1] >> ((cell & 1) * 16)) & 0xFFFFu) - (int)CBIAS;
}

// tpa = voter threads per angle.  Votes of a batch are applied by all voter threads at once with
// shared-memory atomics (order-free); a vote that sees its bin at or above the threshold flags the
// bin, and the exact first triggering point is then recovered per flagged bin by replaying only that
// bin over the batch (counts inside a batch are monotone, so no other bin can trigger earlier).
#ifdef LANE_PPHT_PROF
// schedule probe (make prof; LANE_B200_PPHT_PROF=1): per frame the SM of rank 0, %globaltimer at the start and the end of the
// cluster and thread 0's cycle accounting, written to a global array (printf inside the kernel would distort the schedule)
// and printed by a one-thread kernel behind the launch.  tools/ppht_prof.py drives it; profiles/r2_ppht_schedule.txt.
__device__ unsigned long long g_ppht_prof[8192][8];
__global__ void k4_prof_dump(int n)
{
    for (int f = 0; f < n && f < 8192; f++)
        printf("GT f=%d sm=%llu start=%llu end=%llu vote=%llu xchg=%llu walk=%llu total=%llu\n", f, g_ppht_prof[f][2],
               g_ppht_prof[f][0], g_ppht_prof[f][1], g_ppht_prof[f][3], g_ppht_prof[f][4], g_ppht_prof[f][5], g_ppht_prof[f][6]);
}
#endif

__global__ void __launch_bounds__(416, 2) k4_ppht_v3(const uint32_t *__restrict__ points_all, const int *__restrict__ n_points,
                           const uint32_t *__restrict__ pmask_all, uint32_t *__restrict__ pmask_work,
                           uint32_t *__restrict__ over_all,
                           const int2 *__restrict__ win, int cells_max, int list_cap, int over_cap, int G, int nvw, int tpa,
                           int32_t *__restrict__ lines_all, int *__restrict__ n_lines, LaneGeom g, LaneHoughParams hp, int prof,
                           const int *__restrict__ order)
{
    extern __shared__ __align__(16) unsigned char dyn[];
    uint32_t *cells32 = reinterpret_cast<uint32_t *>(dyn);
    uint32_t *s_list = reinterpret_cast<uint32_t *>(dyn + (((size_t)cells_max * 2 + 15) & ~(size_t)15));
    __shared__ uint32_t s_buf[2][BATCH3];
    __shared__ uint32_t s_rnd[BATCH3];
    __shared__ float s_fx[BATCH3], s_fy[BATCH3];     // batch points as float32, converted once
    __shared__ uint32_t s_hit[HITS_CAP];
    __shared__ XchgSlots s_slots;
    __shared__ int s_trig, s_nflag;
    __shared__ int s_flag_cell[FLAG_CAP], s_flag_slot[FLAG_CAP];
    __shared__ int s_redkey[32];
    __shared__ int s_end[2][2];
    __shared__ int s_nsteps[2];
    __shared__ int s_good;
    __shared__ int s_nhits;
    __shared__ unsigned s_whit[2][24], s_wib[2][24];   // pass-1 ballots of one round, per direction
    __shared__ int s_wlast[2], s_wdone[2], s_wrounds[2];
    __shared__ WalkSetup s_walk;

    unsigned rank;
    asm("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
    const int NVT = nvw * 32;                      // voter threads
    // clusters start in launch order as earlier ones retire: handing out the frames with the most points first keeps the
    // longest sequential loops off the tail of the launch (order = k4_order's permutation; results do not depend on it)
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, f = order ? order[blockIdx.x / G] : blockIdx.x / G;
    const bool producer = wid == nvw;
    const int slot = tid / tpa, sub = tid - slot * tpa;
    const int angle = slot * G + (int)rank;
    const bool active = !producer && angle < LANE_NUM_ANGLES;
    const int WW = (g.W + 31) / 32;
    const int mask_words = g.bh * WW;
    uint32_t *pm = pmask_work + ((size_t)f * G + rank) * mask_words;
    const float cs = active ? c_ppht_cos[angle] : 0.f, sn = active ? c_ppht_sin[angle] : 0.f;
    const int2 wn = active ? win[angle] : make_int2(0, 0);
    const int cell0 = wn.y - wn.x;                 // cell of rho r = cell0 + r

    for (int i = tid; i < cells_max / 2; i += blockDim.x) cells32[i] = CBIAS | (CBIAS << 16);
    {   // private copy of the frame's mask (walks clear bits in it)
        const uint4 *src = reinterpret_cast<const uint4 *>(pmask_all + (size_t)f * mask_words);
        uint4 *dst = reinterpret_cast<uint4 *>(pm);
        const int n4 = mask_words / 4;             // rows are padded so mask_words % 4 == 0 (launcher checks)
        int i = tid;
        for (; i + 3 * (int)blockDim.x < n4; i += 4 * blockDim.x) {
            uint4 a = src[i], b = src[i + blockDim.x], c = src[i + 2 * blockDim.x], d = src[i + 3 * blockDim.x];
            dst[i] = a; dst[i + blockDim.x] = b; dst[i + 2 * blockDim.x] = c; dst[i + 3 * blockDim.x] = d;
        }
        for (; i < n4; i += blockDim.x) dst[i] = src[i];
    }
    if (tid < 32) { s_slots.v[0][tid & 15] = 0; s_slots.v[1][tid & 15] = 0; }
    const int count0 = n_points[f];
    const uint32_t *glist = points_all + (size_t)f * g.max_points;
    // The list lives in shared memory up to list_cap points; a longer one (every 4K generator frame: 3.3 k points)
    // continues in this CTA's private global extension.  Swap-remove only ever touches a random index and the current
    // tail, so once the list has shrunk below list_cap everything is in shared memory again.
    uint32_t *over = over_all + ((size_t)f * G + rank) * over_cap;
    const bool dense = count0 > list_cap + over_cap || (count0 > list_cap && !over_all);   // left to v2
    if (!dense) {
        for (int i = tid; i < min(count0, list_cap); i += blockDim.x) s_list[i] = glist[i];
        for (int i = list_cap + tid; i < count0; i += blockDim.x) __stcg(&over[i - list_cap], glist[i]);
    }
    const bool has_over = !dense && count0 > list_cap;
    const int n_batches = (count0 + BATCH3 - 1) / BATCH3;
    uint64_t rng = 0xFFFFFFFFFFFFFFFFull;
    int remaining = count0, nl = 0;
    unsigned seq = 0;
#ifdef LANE_PPHT_PROF   // cycle accounting of thread 0 (build with -DLANE_PPHT_PROF, run with LANE_B200_PPHT_PROF=1)
    long long tA = 0, tB = 0, tC = 0, tD = 0, tE = 0, tG = 0, tH = 0, tI = 0, t0 = 0, tStart = clock64();
    unsigned long long gt_start;
    unsigned prof_sm;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt_start));
    asm volatile("mov.u32 %0, %%smid;" : "=r"(prof_sm));
    int nTrig = 0, nIter = 0;
#define TICK(acc) do { if (prof && tid == 0) { long long now_ = clock64(); acc += now_ - t0; t0 = now_; } } while (0)
#define PROF(x) x
#else
#define TICK(acc) do { } while (0)
#define PROF(x)
#endif
    __syncthreads();
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
    if (dense) {
        if (tid == 0 && rank == 0) n_lines[f] = -1;
        asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
        return;
    }

    auto bar_v = [&]() { asm volatile("bar.sync 1, %0;" ::"r"(NVT) : "memory"); };
    // Producer warp: draw the next min(BATCH3, remaining) points.  The generator is a serial chain (lane 0),
    // the 64 remainders are independent (all lanes), and the swap-remove on the list runs four steps at a time
    // with the values a later step would have read forwarded in registers.
    auto draw_impl = [&](uint32_t *buf, auto over_tag) {
        // OVER = false (the usual case) keeps the list accesses plain shared-memory loads and stores
        constexpr bool OVER = decltype(over_tag)::value;
        auto lget = [&](int i) -> uint32_t {
            if constexpr (OVER) return i < list_cap ? s_list[i] : __ldcg(&over[i - list_cap]);
            else return s_list[i];
        };
        auto lset = [&](int i, uint32_t v) {
            if constexpr (OVER) { if (i < list_cap) s_list[i] = v; else __stcg(&over[i - list_cap], v); }
            else s_list[i] = v;
        };
        const int P = remaining < BATCH3 ? remaining : BATCH3;
        if (lane == 0) {
            for (int k = 0; k < P; k++) {
                rng = (uint64_t)(uint32_t)rng * 4164903690ull + (uint32_t)(rng >> 32);
                s_rnd[k] = (uint32_t)rng;
            }
        }
        __syncwarp();
        for (int k = lane; k < P; k += 32) s_rnd[k] = s_rnd[k] % (uint32_t)(remaining - k);
        __syncwarp();
        if (lane == 0) {
            int k = 0;
            for (; k + 4 <= P; k += 4) {
                const int i0 = s_rnd[k], i1 = s_rnd[k + 1], i2 = s_rnd[k + 2], i3 = s_rnd[k + 3];
                const int l0 = remaining - k - 1, l1 = l0 - 1, l2 = l0 - 2, l3 = l0 - 3;
                uint32_t a0 = lget(i0), a1 = lget(i1), a2 = lget(i2), a3 = lget(i3);
                uint32_t b0 = lget(l0), b1 = lget(l1), b2 = lget(l2), b3 = lget(l3);
                // step 0 writes list[i0] = b0; later reads of slot i0 must see it, and so on down the chain
                if (i1 == i0) a1 = b0;
                if (l1 == i0) b1 = b0;
                if (i2 == i1) a2 = b1; else if (i2 == i0) a2 = b0;
                if (l2 == i1) b2 = b1; else if (l2 == i0) b2 = b0;
                if (i3 == i2) a3 = b2; else if (i3 == i1) a3 = b1; else if (i3 == i0) a3 = b0;
                if (l3 == i2) b3 = b2; else if (l3 == i1) b3 = b1; else if (l3 == i0) b3 = b0;
                buf[k] = a0; buf[k + 1] = a1; buf[k + 2] = a2; buf[k + 3] = a3;
                lset(i0, b0); lset(i1, b1); lset(i2, b2); lset(i3, b3);       // in order: later steps win
            }
            for (; k < P; k++) {
                const int i = s_rnd[k], l = remaining - k - 1;
                buf[k] = lget(i);
                lset(i, lget(l));
            }
        }
        remaining -= P;
        __syncwarp();
    };
    auto draw = [&](uint32_t *buf) {
        if (has_over) draw_impl(buf, std::true_type{}); else draw_impl(buf, std::false_type{});
    };
    if (producer && n_batches > 0) draw(s_buf[0]);
    __syncthreads();

    for (int bi = 0; bi < n_batches; bi++) {
        uint32_t *batch = s_buf[bi & 1];
        const int P = min(BATCH3, count0 - bi * BATCH3);
        if (producer) {
            if (bi + 1 < n_batches) draw(s_buf[(bi + 1) & 1]);
        } else {
            int k0 = 0;
            PROF(if (prof && tid == 0) t0 = clock64();)
            while (k0 < P) {
                PROF(nIter++;)
                for (int k = k0 + tid; k < P; k += NVT) {            // drop points an earlier walk removed
                    const uint32_t pt = batch[k];
                    if (pt != SKIP) {
                        const int x = pt & 0xFFFF, y = pt >> 16;
                        s_fx[k] = (float)x; s_fy[k] = (float)y;
                        if (!((__ldcg(&pm[(y - g.by0) * WW + (x >> 5)]) >> (x & 31)) & 1u)) batch[k] = SKIP;
                    }
                }
                if (tid == 0) { s_trig = BATCH3; s_nflag = 0; }
                bar_v();
                TICK(tA);
                if (active) {                                         // order-free votes, all voter threads
                    for (int kk = k0 + sub; kk < P; kk += 8 * tpa) {   // eight atomics in flight per thread
                        int c[8], v[8];
#pragma unroll
                        for (int u = 0; u < 8; u++) {
                            const int k = kk + u * tpa;
                            v[u] = -0x40000000;
                            if (k < P && batch[k] != SKIP) {
                                c[u] = cell0 + rho_f(s_fx[k], s_fy[k], cs, sn);
                                v[u] = scell_add(cells32, c[u], 1);
                            }
                        }
#pragma unroll
                        for (int u = 0; u < 8; u++)
                            if (v[u] + 1 >= hp.threshold) {
                                const int i = atomicAdd(&s_nflag, 1);
                                if (i < FLAG_CAP) { s_flag_cell[i] = c[u]; s_flag_slot[i] = slot; }
                            }
                    }
                }
                bar_v();
                TICK(tB);
                const int nflag = s_nflag;
                if (nflag > FLAG_CAP) {
                    // too many flagged bins to replay one by one: redo this batch in point order, one thread per angle
                    if (active)
                        for (int k = k0 + sub; k < P; k += tpa) {
                            const uint32_t pt = batch[k];
                            if (pt != SKIP) scell_add(cells32, cell0 + rho_of(pt & 0xFFFF, pt >> 16, cs, sn), -1);
                        }
                    bar_v();
                    if (active && sub == 0) {
                        int first = BATCH3;
                        for (int k = k0; k < P; k++) {
                            const uint32_t pt = batch[k];
                            if (pt == SKIP) continue;
                            if (scell_add(cells32, cell0 + rho_of(pt & 0xFFFF, pt >> 16, cs, sn), 1) + 1 >= hp.threshold)
                                first = min(first, k);
                        }
                        if (first < BATCH3) atomicMin(&s_trig, first);
                    }
                    bar_v();
                } else if (nflag > 0) {
                    for (int e = wid; e < nflag; e += nvw) {          // one warp replays one flagged bin over the batch
                        const int c = s_flag_cell[e], an = s_flag_slot[e] * G + (int)rank;
                        const float ecs = c_ppht_cos[an], esn = c_ppht_sin[an];
                        const int2 ew = win[an];
                        const int ec0 = ew.y - ew.x;
                        unsigned bal[BATCH3 / 32];
                        int total = 0;
#pragma unroll
                        for (int gq = 0; gq < BATCH3 / 32; gq++) {
                            const int k = gq * 32 + lane;
                            const bool m = k >= k0 && k < P && batch[k] != SKIP && ec0 + rho_f(s_fx[k], s_fy[k], ecs, esn) == c;
                            bal[gq] = __ballot_sync(0xffffffffu, m);
                            total += __popc(bal[gq]);
                        }
                        int need = hp.threshold - (scell_get(cells32, c) - total);   // votes until the bin reaches the threshold
                        if (need < 1) need = 1;                       // already there: its first vote triggers
                        int first = BATCH3;
#pragma unroll
                        for (int gq = 0; gq < BATCH3 / 32; gq++) {
                            const int pc = __popc(bal[gq]);
                            if (first == BATCH3) {
                                if (need <= pc) first = gq * 32 + (int)__fns(bal[gq], 0, need);
                                else need -= pc;
                            }
                        }
                        if (lane == 0 && first < BATCH3) atomicMin(&s_trig, first);
                    }
                    bar_v();
                }
                TICK(tC);
                if (G > 1) {
                    if (tid == 0) s_trig = (int)cluster_reduce(&s_slots, seq, G, rank, (uint32_t)s_trig, 0);
                    bar_v();
                }
                TICK(tD);
                const int t = s_trig;
                if (t == BATCH3) break;
                PROF(nTrig++;)
                int key = 0;                                          // (value, -angle) packed for a max-reduce
                if (active) {
                    for (int k = t + 1 + sub; k < P; k += tpa)        // roll back the votes behind the trigger
                        if (batch[k] != SKIP) scell_add(cells32, cell0 + rho_f(s_fx[k], s_fy[k], cs, sn), -1);
                }
                bar_v();
                if (active && sub == 0) {
                    const uint32_t tp = batch[t];
                    const int v = scell_get(cells32, cell0 + rho_of(tp & 0xFFFF, tp >> 16, cs, sn));
                    key = ((v + 0x8000) << 8) | (255 - angle);
                }
                for (int o = 16; o; o >>= 1) key = max(key, __shfl_xor_sync(0xffffffffu, key, o));
                if (lane == 0) s_redkey[wid] = key;
                bar_v();
                if (tid == 0) {
                    int best = s_redkey[0];
                    for (int w = 1; w < nvw; w++) best = max(best, s_redkey[w]);
                    if (G > 1) best = (int)cluster_reduce(&s_slots, seq, G, rank, (uint32_t)best, 1);
                    const int mn = 255 - (best & 0xFF);
                    const uint32_t tp = batch[t];
                    const int px = tp & 0xFFFF, py = tp >> 16;
                    float a = -c_ppht_sin[mn], b = c_ppht_cos[mn];
                    WalkSetup w;
                    w.x0 = px; w.y0 = py;
                    if (fabsf(a) > fabsf(b)) {
                        w.xflag = 1;
                        w.dx0 = a > 0 ? 1 : -1;
                        w.dy0 = __float2int_rn(__fdiv_rn(__fmul_rn(b, 65536.0f), fabsf(a)));
                        w.y0 = (py << 16) + 32768;
                    } else {
                        w.xflag = 0;
                        w.dy0 = b > 0 ? 1 : -1;
                        w.dx0 = __float2int_rn(__fdiv_rn(__fmul_rn(a, 65536.0f), fabsf(b)));
                        w.x0 = (px << 16) + 32768;
                    }
                    s_walk = w;
                }
                bar_v();
                TICK(tE);
                const WalkSetup w = s_walk;
                // ---- pass 1: half of the voter warps per direction; WSTEPS steps of the line are fetched in one
                // round (every thread issues its loads back to back), ballots go to shared memory, and one lane then
                // runs cv2's gap logic over the bit string.  Lines longer than a round simply take another round.
                {
                    const int half = nvw >= 2 ? nvw / 2 : 1;          // warps per direction
                    const int kdir = nvw >= 2 ? (wid < half ? 0 : (wid < 2 * half ? 1 : 2)) : 0;
                    const int ndir_pass = nvw >= 2 ? 1 : 2;           // a single voter warp does the directions one after the other
                    for (int dp = 0; dp < ndir_pass; dp++) {
                        const int k = nvw >= 2 ? kdir : dp;
                        const int wl = nvw >= 2 ? (wid - k * half) : 0;   // warp index inside the direction group
                        const int gsteps = half * 32 * WPT;
                        if (tid < 2) { s_wlast[tid] = 0; s_wdone[tid] = 0; s_wrounds[tid] = 0; }
                        bar_v();
                        for (int base = 0;; base += gsteps) {
                            if (k < 2 && !s_wdone[k]) {
                                unsigned hb[WPT], ibb[WPT];
                                // all WPT mask words are requested before any is looked at (one L2 round trip, not WPT)
                                int sh[WPT];
                                bool ibv[WPT], roi[WPT];
                                uint32_t mw[WPT];
#pragma unroll
                                for (int j = 0; j < WPT; j++) {
                                    int j1, i1;
                                    step_pixel(w, k, base + (wl * WPT + j) * 32 + lane, j1, i1);
                                    ibv[j] = j1 >= 0 && j1 < g.W && i1 >= 0 && i1 < g.H;
                                    roi[j] = ibv[j] && i1 >= g.by0 && i1 < g.by1;
                                    sh[j] = j1 & 31;
                                    mw[j] = __ldcg(&pm[roi[j] ? (i1 - g.by0) * WW + (j1 >> 5) : 0]);
                                }
#pragma unroll
                                for (int j = 0; j < WPT; j++) {
                                    ibb[j] = __ballot_sync(0xffffffffu, ibv[j]);
                                    hb[j] = __ballot_sync(0xffffffffu, roi[j] && ((mw[j] >> sh[j]) & 1u));
                                }
                                if (lane == 0)
#pragma unroll
                                    for (int j = 0; j < WPT; j++) { s_whit[k][wl * WPT + j] = hb[j]; s_wib[k][wl * WPT + j] = ibb[j]; }
                            }
                            bar_v();
                            const bool warp_gap = nvw >= 2 && hp.max_gap >= 31;       // a word per lane, see below
                            if (warp_gap && wid < 2 && !s_wdone[wid]) {
                                // cv2's gap logic over this round's bit string, a 32-step word per lane: with max_gap >= 31
                                // only the distance from the last hit before a word to the word's first hit (and to the
                                // word's end) can stop the walk, and "last hit so far" is a prefix maximum
                                const int kk = wid, nq = half * WPT, NONE = -0x40000000;
                                unsigned Hh = lane < nq ? s_whit[kk][lane] : 0u;
                                const unsigned IB = lane < nq ? s_wib[kk][lane] : 0xFFFFFFFFu;
                                const int limit = (~IB) ? __ffs(~IB) - 1 : 32;
                                if (limit < 32) Hh &= (1u << limit) - 1u;
                                const int b32 = base + 32 * lane;
                                const int lastpos = Hh ? b32 + 31 - __clz(Hh) : NONE;
                                int run = lastpos;
                                for (int o2 = 1; o2 < 32; o2 <<= 1) {
                                    const int t2 = __shfl_up_sync(0xffffffffu, run, o2);
                                    if (lane >= o2) run = max(run, t2);
                                }
                                int last_in = __shfl_up_sync(0xffffffffu, run, 1);
                                if (lane == 0) last_in = NONE;
                                last_in = max(last_in, s_wlast[kk]);
                                const bool c1 = Hh && (b32 + __ffs(Hh) - 1 - last_in > hp.max_gap + 1);
                                const int last_out = (Hh && !c1) ? lastpos : last_in;
                                const bool c2 = !c1 && (limit < 32 || b32 + 31 - last_out > hp.max_gap);
                                const unsigned db = __ballot_sync(0xffffffffu, lane < nq && (c1 || c2));
                                const int q = db ? __ffs(db) - 1 : nq - 1;
                                const int last = __shfl_sync(0xffffffffu, (db && c1) ? last_in : last_out, q);
                                if (lane == 0) {
                                    s_wrounds[kk]++;
                                    s_wlast[kk] = last;
                                    if (db) {
                                        s_wdone[kk] = 1;
                                        int j1, i1;
                                        step_pixel(w, kk, last, j1, i1);
                                        s_end[kk][0] = j1; s_end[kk][1] = i1;
                                        s_nsteps[kk] = last + 1;
                                    }
                                }
                            }
                            if (!warp_gap && tid < 2 && !s_wdone[tid] && (nvw >= 2 || tid == k)) {   // serial form (short max_gap)
                                const int kk = tid;
                                s_wrounds[kk]++;
                                int last = s_wlast[kk];
                                bool done = false;
                                for (int q = 0; q < half * WPT && !done; q++) {
                                    const int b32 = base + 32 * q;
                                    unsigned Hh = s_whit[kk][q];
                                    const unsigned IB = s_wib[kk][q];
                                    const int limit = (~IB) ? __ffs(~IB) - 1 : 32;
                                    if (limit < 32) Hh &= (1u << limit) - 1u;
                                    if (hp.max_gap >= 31) {           // a gap inside one word can never end the walk
                                        if (Hh) {
                                            if (b32 + __ffs(Hh) - 1 - last > hp.max_gap + 1) done = true;
                                            else last = b32 + 31 - __clz(Hh);
                                        }
                                    } else {
                                        while (Hh) {
                                            const int p = b32 + __ffs(Hh) - 1;
                                            if (p - last > hp.max_gap + 1) { done = true; break; }
                                            last = p;
                                            Hh &= Hh - 1;
                                        }
                                    }
                                    if (!done) {
                                        if (limit < 32) done = true;
                                        else if (b32 + 31 - last > hp.max_gap) done = true;
                                    }
                                }
                                s_wlast[kk] = last;
                                if (done) {
                                    s_wdone[kk] = 1;
                                    int j1, i1;
                                    step_pixel(w, kk, last, j1, i1);
                                    s_end[kk][0] = j1; s_end[kk][1] = i1;
                                    s_nsteps[kk] = last + 1;
                                }
                            }
                            bar_v();
                            if (nvw >= 2 ? (s_wdone[0] && s_wdone[1]) : s_wdone[k]) break;
                        }
                    }
                }
                TICK(tG);
                if (tid == 0) {
                    int good = abs(s_end[1][0] - s_end[0][0]) >= hp.min_len || abs(s_end[1][1] - s_end[0][1]) >= hp.min_len;
                    s_good = good;
                    if (good) {
                        if (rank == 0 && nl < g.max_segments) {
                            int32_t *lines = lines_all + (size_t)f * g.max_segments * 4;
                            lines[4 * nl + 0] = s_end[0][0]; lines[4 * nl + 1] = s_end[0][1];
                            lines[4 * nl + 2] = s_end[1][0]; lines[4 * nl + 3] = s_end[1][1];
                        }
                        nl++;
                    }
                }
                {                                                     // pass 2: clear, and un-vote if good
                    // both directions share the rounds: virtual step v < ns0 is step v of direction 0, the rest belong
                    // to direction 1 (whose step 0 is the trigger pixel again and is left to direction 0)
                    const int ns0 = s_nsteps[0], nst = ns0 + s_nsteps[1];
                    const bool bits0 = s_wrounds[0] == 1, bits1 = s_wrounds[1] == 1;
                    const int per_round = min(4 * NVT, HITS_CAP);
                    for (int base = 0; base < nst; base += per_round) {
                        if (tid == 0) s_nhits = 0;
                        bar_v();
                        // A walk that fit one pass-1 round left its hit bits in shared memory: they are exactly the set
                        // mask pixels along the line (the private mask has not changed since), so the mask is cleared
                        // with fire-and-forget atomics and nothing is read back.  Longer walks probe the mask again.
                        for (int v = base + tid; v < min(nst, base + per_round); v += NVT) {
                            const int k = v >= ns0 ? 1 : 0, s = k ? v - ns0 : v;
                            if (k == 1 && s == 0) continue;
                            int j1, i1;
                            if (k ? bits1 : bits0) {
                                if ((s_whit[k][s >> 5] >> (s & 31)) & 1u) {
                                    step_pixel(w, k, s, j1, i1);
                                    atomicAnd(&pm[(i1 - g.by0) * WW + (j1 >> 5)], ~(1u << (j1 & 31)));
                                    const int h = atomicAdd(&s_nhits, 1);
                                    s_hit[h] = ((uint32_t)i1 << 16) | (uint32_t)j1;
                                }
                                continue;
                            }
                            step_pixel(w, k, s, j1, i1);
                            if (i1 >= g.by0 && i1 < g.by1 && j1 >= 0 && j1 < g.W) {
                                const uint32_t bit = 1u << (j1 & 31);
                                if (atomicAnd(&pm[(i1 - g.by0) * WW + (j1 >> 5)], ~bit) & bit) {
                                    const int h = atomicAdd(&s_nhits, 1);
                                    s_hit[h] = ((uint32_t)i1 << 16) | (uint32_t)j1;
                                }
                            }
                        }
                        bar_v();
                        if (s_good && active) {
                            const int nh = s_nhits;
                            for (int h = sub; h < nh; h += tpa) {
                                const uint32_t p = s_hit[h];
                                scell_add(cells32, cell0 + rho_f((float)(p & 0xFFFFu), (float)(p >> 16), cs, sn), -1);
                            }
                        }
                        bar_v();
                    }
                }
                TICK(tH);
                k0 = t + 1;
            }
        }
        PROF(if (prof && tid == 0) t0 = clock64();)
        __syncthreads();
        TICK(tI);
    }
#ifdef LANE_PPHT_PROF
    if (prof && tid == 0 && rank == 0 && f < 8192) {
        unsigned long long gt_end;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt_end));
        g_ppht_prof[f][0] = gt_start; g_ppht_prof[f][1] = gt_end; g_ppht_prof[f][2] = prof_sm;
        g_ppht_prof[f][3] = tB; g_ppht_prof[f][4] = tD + tE; g_ppht_prof[f][5] = tG + tH; g_ppht_prof[f][6] = clock64() - tStart;
    }
#endif
    if (tid == 0 && rank == 0) n_lines[f] = nl;
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// order[k] = index of the frame with the k-th largest point count (ties by index): longest-processing-time-first for the
// frame-per-cluster kernels.  n is a batch (hundreds of frames): a rank sort.
__global__ void k4_order(const int *__restrict__ n_points, int *__restrict__ order, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int mine = n_points[i];
    int rank = 0;
    for (int j = 0; j < n; j++) {
        const int o = __ldg(&n_points[j]);
        rank += (o > mine) || (o == mine && j < i);
    }
    order[rank] = i;
}

}  // namespace

void launch_ppht_v2(uint32_t *points, const int *n_points, uint32_t *pmask, uint32_t *accum16, const int2 *win,
                    int cells_per_frame, int32_t *lines, int *n_lines, LaneGeom g, LaneHoughParams hp, int n,
                    cudaStream_t st, int *launches, int only_flagged)
{
    if (!only_flagged) cudaMemsetAsync(accum16, 0x40, sizeof(uint16_t) * (size_t)n * cells_per_frame, st);
    k4_ppht_v2<<<n, NT2, 0, st>>>(points, n_points, pmask, accum16, win, cells_per_frame, lines, n_lines, g, hp,
                                  only_flagged);
    *launches += 1;
}

// v3 launch: false if the geometry does not fit (caller uses v2)
bool launch_ppht_v3(const uint32_t *points, const int *n_points, const uint32_t *pmask, uint32_t *pmask_work,
                    uint32_t *list_over, const int2 *win3, int cells_max, int list_cap, int over_cap, int G, int32_t *lines, int *n_lines, LaneGeom g,
                    LaneHoughParams hp, int n, cudaStream_t st, int *launches, int *order)
{
    if (G < 1 || (g.bh * ((g.W + 31) / 32)) % 4 != 0 || ((uintptr_t)pmask % 16) != 0) return false;
    if (order) {
        k4_order<<<(n + 255) / 256, 256, 0, st>>>(n_points, order, n);
        *launches += 1;
    }
    const int angles = (LANE_NUM_ANGLES + G - 1) / G;
    int tpa = 384 / angles;                      // aim at ~12 voter warps per CTA
    tpa = tpa < 1 ? 1 : (tpa > 8 ? 8 : tpa);
    const int nvw = (angles * tpa + 31) / 32;
    const size_t smem = (((size_t)cells_max * 2 + 15) & ~(size_t)15) + sizeof(uint32_t) * (size_t)list_cap;
    static bool configured[LANE_MAX_DEVICES];
    if (!configured[lane_cur_device()]) {
        cudaFuncSetAttribute(k4_ppht_v3, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
        cudaFuncSetAttribute(k4_ppht_v3, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
        configured[lane_cur_device()] = true;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(n * G);
    cfg.blockDim = dim3((nvw + 1) * 32);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = G; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, k4_ppht_v3, points, n_points, pmask, pmask_work, list_over, win3, cells_max, list_cap, over_cap, G, nvw, tpa,
                                       lines, n_lines, g, hp, getenv("LANE_B200_PPHT_PROF") ? 1 : 0, (const int *)order);
    if (e != cudaSuccess) { cudaGetLastError(); return false; }
#ifdef LANE_PPHT_PROF
    if (getenv("LANE_B200_PPHT_PROF")) k4_prof_dump<<<1, 1, 0, st>>>(n);
#endif
    *launches += 1;
    return true;
}

int lane_ppht_list_cap_v3() { return LIST_CAP3; }
int lane_ppht_over_cap_v3() { return OVER_CAP3; }

// Plan the v3 layout: smallest cluster size whose per-CTA cell count fits shared memory.  win3[n] = (rmin_n,
// first cell inside CTA n % G).  Returns G (0 if nothing fits) and *cells_max.
int lane_ppht_plan_v3(const int2 *win, int cells_total, int2 *win3, int *cells_max, int *list_cap)
{
    int width[LANE_NUM_ANGLES];
    for (int n = 0; n < LANE_NUM_ANGLES; n++)
        width[n] = (n + 1 < LANE_NUM_ANGLES ? win[n + 1].y : cells_total) - win[n].y;
    // A smaller cluster means more frames in flight and fewer exchange partners, so a shorter shared point list is
    // accepted when that is all a cluster size lacks (4K: 8 CTAs with 2560 list entries instead of 16 CTAs -- 37 frames in
    // flight instead of 18, 1.76 ms against 3.6 ms per 128 frames; longer lists continue in the global extension).
    static const int caps[3] = {LIST_CAP3, 2560, 2048};
    for (int pass = 0; pass < 2; pass++)
    for (int G = 1; G <= 16; G *= 2) {
        const size_t budget = pass == 0 ? 112 * 1024 : 226 * 1024;   // first try to fit two CTAs per SM
        int off[16] = {0};
        for (int n = 0; n < LANE_NUM_ANGLES; n++) {
            win3[n] = make_int2(win[n].x, off[n % G]);
            off[n % G] += width[n];
        }
        int mx = 0;
        for (int r = 0; r < G; r++) mx = off[r] > mx ? off[r] : mx;
        mx = (mx + 7) & ~7;
        for (int cap : caps)
            if ((size_t)mx * 2 + sizeof(uint32_t) * (size_t)cap + 4700 <= budget) { *cells_max = mx; *list_cap = cap; return G; }
    }
    return 0;
}

// Per-angle rho windows reachable from the ROI mask: extremes of the (monotone) rounded rho over every
// row span of the mask, evaluated with the device's float32 arithmetic.  win[n] = (rmin_n, first cell).
int lane_ppht_windows(const uint8_t *mask, int H, int W, int2 *win)
{
    const float theta = (float)(M_PI / 180.0);
    int rmin[LANE_NUM_ANGLES], rmax[LANE_NUM_ANGLES];
    float pc[LANE_NUM_ANGLES], ps[LANE_NUM_ANGLES];
    for (int n = 0; n < LANE_NUM_ANGLES; n++) {
        pc[n] = (float)cos((double)n * theta); ps[n] = (float)sin((double)n * theta);
        rmin[n] = 0x7fffffff; rmax[n] = -0x7fffffff;
    }
    auto eval = [&](int x, int y) {
        for (int n = 0; n < LANE_NUM_ANGLES; n++) {
            volatile float a = (float)x * pc[n];
            volatile float b = (float)y * ps[n];
            int r = (int)lrintf(a + b);
            if (r < rmin[n]) rmin[n] = r;
            if (r > rmax[n]) rmax[n] = r;
        }
    };
    for (int y = 0; y < H; y++) {
        const uint8_t *row = mask + (size_t)y * W;
        for (int x = 0; x < W; x++)
            if (row[x] && (x == 0 || !row[x - 1] || x == W - 1 || !row[x + 1])) eval(x, y);
    }
    int cells = 0;
    for (int n = 0; n < LANE_NUM_ANGLES; n++) {
        if (rmax[n] < rmin[n]) { rmin[n] = 0; rmax[n] = 0; }
        win[n] = make_int2(rmin[n], cells);
        cells += (rmax[n] - rmin[n] + 1 + 1) & ~1;      // rows start on word boundaries
    }
    return cells;
}
