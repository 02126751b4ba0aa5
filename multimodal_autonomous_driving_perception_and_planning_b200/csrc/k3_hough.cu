// K3: standard Hough accumulator + local-maximum peaks (BASELINE.json north-star kernel #3; what
// cv2.HoughLines(masked, 1, pi/180, thr) votes into and returns -- SURVEY.md A.5).  The reference's detect() never
// builds it, so it is an add-on that runs on demand on the frames of the last batch.
//   rho = rint(float(x)*cos + float(y)*sin) in float32 without FMA, tables accumulated in float32 (they differ from
//   the HoughLinesP tables); peaks: v > thr, v > left, v >= right, v > previous angle, v >= next angle; output order:
//   votes descending, ties by ascending flat index of the padded accumulator.
//
// k3_batch (whole batch, no debug mode needed): grid = (theta band, frame).  A CTA keeps the 16-bit rho rows of its band
// of angles -- plus the two neighbouring angles its peak test needs -- in shared memory, scans the ROI rows of the
// frame's edge bit-plane (edge & ROI words, so it does not depend on the point list the PPHT consumes), compacts the
// set pixels into a shared chunk and votes them: a warp takes one angle and 32 consecutive points, lanes that hit the
// same cell are merged with match.any and the leader adds their count with one shared-memory atomic (consecutive edge
// pixels of a row share their cell for the near-horizontal angles).  Then the band's peaks are appended to the frame's
// list and, in verification mode, its rows are written to the padded int32 accumulator.  k3_sort orders each frame's
// list on the device (rank sort; the lists are short).
// k3_accum / k3_peaks: the round-1 one-frame form (one CTA per theta), kept for the single-frame tap.
#include "lane_common.cuh"

#include <math.h>

#include <algorithm>

__constant__ float c_std_cos[LANE_NUM_ANGLES], c_std_sin[LANE_NUM_ANGLES];

void lane_upload_tables_std()
{
    float sc[LANE_NUM_ANGLES], ss[LANE_NUM_ANGLES];
    const float theta = (float)(M_PI / 180.0);
    float ang = 0.0f;       // HoughLines accumulates the angle in float32 (A.5)
    for (int n = 0; n < LANE_NUM_ANGLES; n++) {
        sc[n] = (float)cos((double)ang);
        ss[n] = (float)sin((double)ang);
        ang += theta;
    }
    cudaMemcpyToSymbol(c_std_cos, sc, sizeof(sc));
    cudaMemcpyToSymbol(c_std_sin, ss, sizeof(ss));
}

namespace {

__global__ void __launch_bounds__(256) k3_accum(const uint32_t *__restrict__ points, const int *__restrict__ n_points,
                                                int32_t *__restrict__ accum, int numrho)
{
    extern __shared__ int row[];      // numrho + 2
    const int n = blockIdx.x, tid = threadIdx.x;
    for (int i = tid; i < numrho + 2; i += 256) row[i] = 0;
    __syncthreads();
    const float cs = c_std_cos[n], sn = c_std_sin[n];
    const int off = (numrho - 1) / 2 + 1;
    const int cnt = *n_points;
    for (int i = tid; i < cnt; i += 256) {
        uint32_t pt = points[i];
        int r = __float2int_rn(__fadd_rn(__fmul_rn((float)(pt & 0xFFFF), cs), __fmul_rn((float)(pt >> 16), sn)));
        atomicAdd(&row[r + off], 1);
    }
    __syncthreads();
    int32_t *dst = accum + (size_t)(n + 1) * (numrho + 2);
    for (int i = tid; i < numrho + 2; i += 256) dst[i] = row[i];
}

// peaks: (flat index, votes) of cells that beat threshold and their 4-neighbourhood with cv2's >/>= pattern
__global__ void k3_peaks(const int32_t *__restrict__ accum, int numrho, int threshold, int2 *__restrict__ peaks,
                         int max_peaks, int *__restrict__ n_peaks)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= numrho * LANE_NUM_ANGLES) return;
    int n = i / numrho, r = i - n * numrho;
    int base = (n + 1) * (numrho + 2) + r + 1;
    int v = accum[base];
    if (v > threshold && v > accum[base - 1] && v >= accum[base + 1] && v > accum[base - numrho - 2] &&
        v >= accum[base + numrho + 2]) {
        int pos = atomicAdd(n_peaks, 1);
        if (pos < max_peaks) peaks[pos] = make_int2(base, v);
    }
}

// ---- batched form ----------------------------------------------------------------------------------------
constexpr int K3T = 256;
constexpr int K3_CAP = 2048;           // points per voting round (a quarter of a scan round can never exceed it)

struct K3Args {
    const uint32_t *edge_bits;         // [n][H][WW]
    const uint32_t *roi_bits;          // [R][roi_stride] ROI planes, each [H][WW]
    int32_t *accum;                    // [n][182][numrho+2] or null
    int2 *peaks;                       // [n][max_peaks] (flat padded index, votes), unordered
    int *n_peaks;                      // [n]
    int H, WW, by0, by1, numrho, TB, threshold, max_peaks;
    const int *roi_index;              // [n] ROI plane of each frame, or null: every frame uses plane 0
    size_t roi_stride;
};

__device__ __forceinline__ int k3_cell(const uint32_t *row, int c) { return (int)((row[c >> 1] >> ((c & 1) * 16)) & 0xFFFFu); }

__global__ void __launch_bounds__(K3T) k3_batch(K3Args A)
{
    extern __shared__ __align__(16) uint32_t k3sm[];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, f = blockIdx.y;
    const int a0 = blockIdx.x * A.TB, a1 = min(a0 + A.TB, LANE_NUM_ANGLES);      // angles this CTA owns
    const int R = a1 - a0 + 2;                                                   // rows held: a0-1 .. a1
    const int row_cells = A.numrho + 2, row_words = (row_cells + 1) / 2;
    uint32_t *rows = k3sm;                                                       // [TB+2][row_words] packed u16 cells
    uint32_t *pts = k3sm + (size_t)(A.TB + 2) * row_words;                        // [K3_CAP]
    __shared__ int s_cnt, s_round[2];                   // s_round alternates by scan round (reset one round ahead)
    for (int i = tid; i < R * row_words; i += K3T) rows[i] = 0;
    if (tid == 0) { s_cnt = 0; s_round[0] = 0; s_round[1] = 0; }
    __syncthreads();
    const int off = (A.numrho - 1) / 2 + 1;
    const uint32_t *eb = A.edge_bits + (size_t)f * A.H * A.WW;
    const uint32_t *roi = A.roi_bits + (A.roi_index ? (size_t)A.roi_index[f] * A.roi_stride : 0);
    const int n_words = (A.by1 - A.by0) * A.WW;

    // vote the s_cnt points in pts[]: a warp per angle row, 32 consecutive points per step, equal cells merged
    auto vote = [&]() {
        const int P = s_cnt;
        for (int j = wid; j < R; j += K3T / 32) {
            const int a = a0 - 1 + j;
            if (a < 0 || a >= LANE_NUM_ANGLES) continue;      // cv2's padding rows stay zero
            const float cs = c_std_cos[a], sn = c_std_sin[a];
            uint32_t *row = rows + (size_t)j * row_words;
            for (int p0 = 0; p0 < P; p0 += 32) {
                const int p = p0 + lane;
                const bool valid = p < P;
                const unsigned act = __ballot_sync(0xffffffffu, valid);
                if (valid) {
                    const uint32_t pt = pts[p];
                    const int cell = __float2int_rn(__fadd_rn(__fmul_rn((float)(pt & 0xFFFFu), cs),
                                                              __fmul_rn((float)(pt >> 16), sn))) + off;
                    const unsigned peers = __match_any_sync(act, cell);           // lanes voting the same cell
                    if ((int)(__ffs(peers) - 1) == lane)
                        atomicAdd(&row[cell >> 1], (uint32_t)__popc(peers) << ((cell & 1) * 16));
                }
            }
        }
    };
    auto append = [&](uint32_t m, int y, int w) {            // this thread's set pixels go to the chunk
        if (!m) return;
        int pos = atomicAdd(&s_cnt, __popc(m));
        while (m) {
            pts[pos++] = ((uint32_t)y << 16) | (uint32_t)(w * 32 + __ffs(m) - 1);
            m &= m - 1;
        }
    };
    auto flush = [&]() {                                      // all threads
        __syncthreads();
        vote();
        __syncthreads();
        if (tid == 0) s_cnt = 0;
        __syncthreads();
    };

    // scan the ROI rows of (edge & ROI), a word per thread, in rounds of K3T words
    for (int base = 0, par = 0; base < n_words; base += K3T, par ^= 1) {
        const int i = base + tid;
        uint32_t m = 0;
        int y = 0, w = 0;
        if (i < n_words) {
            y = A.by0 + i / A.WW; w = i % A.WW;
            m = eb[(size_t)y * A.WW + w] & roi[(size_t)y * A.WW + w];
        }
        if (m) atomicAdd(&s_round[par], __popc(m));
        __syncthreads();
        const int rt = s_round[par];
        if (tid == 0) s_round[par ^ 1] = 0;                   // last read a round ago, next used after the barrier below
        __syncthreads();
        if (rt == 0) continue;                                // block-uniform
        if (s_cnt + rt > K3_CAP) flush();                     // s_cnt is stable here (read after a barrier)
        if (rt <= K3_CAP) {
            append(m, y, w);
        } else {                                              // dense round: a quarter of the threads at a time (<= 2048 px)
            for (int q = 0; q < 4; q++) {
                if ((tid >> 6) == q) append(m, y, w);
                flush();
            }
        }
        __syncthreads();
    }
    flush();

    // ---- outputs of the owned angles: peaks, and (verification mode) the padded int32 rows
    for (int j = 1; j < R - 1; j++) {
        const int a = a0 - 1 + j;
        const uint32_t *row = rows + (size_t)j * row_words, *up = row - row_words, *dn = row + row_words;
        const int flat0 = (a + 1) * row_cells;
        if (A.accum) {
            int32_t *dst = A.accum + ((size_t)f * (LANE_NUM_ANGLES + 2) + (a + 1)) * row_cells;
            for (int c = tid; c < row_cells; c += K3T) dst[c] = k3_cell(row, c);
        }
        if (A.peaks) {
            for (int c = 1 + tid; c <= A.numrho; c += K3T) {
                const int v = k3_cell(row, c);
                if (v > A.threshold && v > k3_cell(row, c - 1) && v >= k3_cell(row, c + 1) && v > k3_cell(up, c) &&
                    v >= k3_cell(dn, c)) {
                    const int pos = atomicAdd(&A.n_peaks[f], 1);
                    if (pos < A.max_peaks) A.peaks[(size_t)f * A.max_peaks + pos] = make_int2(flat0 + c, v);
                }
            }
        }
    }
}

// cv2's output order per frame: votes descending, ties by ascending flat index.  Rank sort: entry i goes to the slot
// equal to the number of entries that precede it (flat indices are unique, so the ranks are a permutation).
__global__ void __launch_bounds__(K3T) k3_sort(const int2 *__restrict__ peaks, const int *__restrict__ n_peaks,
                                               int32_t *__restrict__ out, int max_peaks, int numrho)
{
    __shared__ int2 tile[1024];
    const int f = blockIdx.x, tid = threadIdx.x;
    const int m = min(n_peaks[f], max_peaks);
    const int2 *src = peaks + (size_t)f * max_peaks;
    int32_t *dst = out + (size_t)f * max_peaks * 3;
    for (int i0 = 0; i0 < m; i0 += K3T) {
        const int i = i0 + tid;
        const int2 me = i < m ? src[i] : make_int2(0, 0);
        int rank = 0;
        for (int t0 = 0; t0 < m; t0 += 1024) {
            __syncthreads();
            for (int t = tid; t < min(1024, m - t0); t += K3T) tile[t] = src[t0 + t];
            __syncthreads();
            if (i < m) {
                const int tn = min(1024, m - t0);
                for (int t = 0; t < tn; t++) {
                    const int2 o = tile[t];
                    rank += (o.y > me.y) || (o.y == me.y && o.x < me.x);
                }
            }
        }
        if (i < m) {
            const int nn = me.x / (numrho + 2) - 1, r = me.x - (nn + 1) * (numrho + 2) - 1;
            dst[3 * rank] = r; dst[3 * rank + 1] = nn; dst[3 * rank + 2] = me.y;
        }
    }
}

}  // namespace

void launch_hough_accum(const uint32_t *points, const int *n_points, int32_t *accum_padded, LaneGeom g,
                        cudaStream_t st)
{
    size_t smem = sizeof(int) * (g.numrho + 2);
    cudaFuncSetAttribute(k3_accum, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    cudaMemsetAsync(accum_padded, 0, sizeof(int32_t) * (size_t)(LANE_NUM_ANGLES + 2) * (g.numrho + 2), st);
    k3_accum<<<LANE_NUM_ANGLES, 256, smem, st>>>(points, n_points, accum_padded, g.numrho);
}

void launch_hough_peaks(const int32_t *accum_padded, int numrho, int threshold, int2 *peaks, int max_peaks,
                        int *n_peaks, cudaStream_t st)
{
    cudaMemsetAsync(n_peaks, 0, sizeof(int), st);
    int total = numrho * LANE_NUM_ANGLES;
    k3_peaks<<<(total + 255) / 256, 256, 0, st>>>(accum_padded, numrho, threshold, peaks, max_peaks, n_peaks);
}

// Batched standard Hough over the n frames whose edge planes are in edge_bits.  accum (optional) receives the padded
// int32 accumulators [n][182][numrho+2]; peaks_sorted [n][max_peaks][3] = (rho index, angle index, votes) in cv2 order,
// n_peaks[n] = peaks found (may exceed max_peaks; only that many are kept).  peaks_tmp: [n][max_peaks] int2 scratch.
bool launch_hough_batch(const uint32_t *edge_bits, const uint32_t *roi_bits, const int *roi_index, size_t roi_stride,
                        int32_t *accum, int2 *peaks_tmp, int32_t *peaks_sorted, int *n_peaks, LaneGeom g, int threshold,
                        int max_peaks, int n, cudaStream_t st)
{
    const int row_words = (g.numrho + 2 + 1) / 2;
    const size_t row_bytes = (size_t)row_words * 4, fixed = sizeof(uint32_t) * K3_CAP;
    // angles per CTA: as many rows as fit ~100 KB (two CTAs per SM), at least 2 owned angles; two of the rows are halo
    int rows = (int)((100 * 1024 - fixed) / row_bytes);
    if (rows < 4) rows = (int)((220 * 1024 - fixed) / row_bytes);
    if (rows < 3) return false;
    const int TB = std::min(rows - 2, 30);
    const size_t smem = (size_t)(TB + 2) * row_bytes + fixed;
    static bool configured[LANE_MAX_DEVICES];
    if (!configured[lane_cur_device()]) {
        cudaFuncSetAttribute(k3_batch, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
        configured[lane_cur_device()] = true;
    }
    K3Args A{};
    A.edge_bits = edge_bits; A.roi_bits = roi_bits; A.roi_index = roi_index; A.roi_stride = roi_stride; A.accum = accum; A.peaks = peaks_tmp; A.n_peaks = n_peaks;
    A.H = g.H; A.WW = (g.W + 31) / 32; A.by0 = g.by0; A.by1 = g.by1; A.numrho = g.numrho; A.TB = TB;
    A.threshold = threshold; A.max_peaks = max_peaks;
    cudaMemsetAsync(n_peaks, 0, sizeof(int) * n, st);
    if (accum) {        // cv2's padding rows (angle -1 and 180) are zero; the inner rows are written by the kernel
        const size_t row = (size_t)(g.numrho + 2), frame = row * (LANE_NUM_ANGLES + 2);
        for (int f = 0; f < n; f++) {
            cudaMemsetAsync(accum + f * frame, 0, sizeof(int32_t) * row, st);
            cudaMemsetAsync(accum + f * frame + (LANE_NUM_ANGLES + 1) * row, 0, sizeof(int32_t) * row, st);
        }
    }
    dim3 grid((LANE_NUM_ANGLES + TB - 1) / TB, n);
    k3_batch<<<grid, K3T, smem, st>>>(A);
    if (peaks_sorted) k3_sort<<<n, K3T, 0, st>>>(peaks_tmp, n_peaks, peaks_sorted, max_peaks, g.numrho);
    return cudaPeekAtLastError() == cudaSuccess;
}
