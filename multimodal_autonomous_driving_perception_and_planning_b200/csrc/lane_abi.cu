// C-ABI shim over the lane-detection kernels: context, device buffers, stage sequencing.
// Entry points are declared (with the reference lines they replace) in include/lane_b200.h.
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "cuda_owned.h"
#include "k0_common.cuh"

#define LANE_COPY_EVENTS 8

static thread_local std::string g_create_error;
void lane_set_global_error(const char *msg) { g_create_error = msg ? msg : ""; }

#include "host_stage.h"

struct lane_ctx {
    int device = 0;
    int max_batch = 0;
    LaneGeom g{};
    LaneHoughParams hp{50, 50, 150};
    double smooth = 0.7, one_minus_smooth = 1 - 0.7;
    bool have_roi = false, have_lut = false, debug = false, profiling = false;
    int blur = 1;                     // 0: Canny runs on the plain grayscale plane (lane_set_preprocess)
    CudaStream st, copy_st;           // compute stream (or the caller's, lane_ctx_set_stream); H2D stream for chunked host batches
    // Second compute stream for the back half of the path (PPHT + fit + record copies) of device-resident batches: the
    // PPHT kernel runs in waves of whole frames (71 clusters at 1080p) and its last wave leaves 40 % of the SMs idle for a
    // frame's latency; with the edge kernels of the NEXT queued batch on the first stream those SMs are used.  The buffers
    // that cross from the edge half to the back half are kept per result slot (see `two`).
    CudaStream st2;
    CudaEvent edge_done[2];
    bool overlap_now = false;                       // the batch being enqueued runs its back half on st2
    CudaEvent copy_ev[LANE_COPY_EVENTS], start_ev;
    std::string err;

    // device buffers
    DeviceArray<uint8_t> d_frames;    // staging for host frames / BGR output of the ingest kernels (lazy)
    DeviceArray<uint8_t> d_src;       // staging for host frames the ingest kernels convert / resize (lazy, grows)
    DeviceArray<RigFrame> d_rig;      // [2][B] frame descriptors of rig batches, per result slot (lazy)
    DeviceArray<uint8_t> d_blur;      // blurred plane: unfused path and verification taps only (lazy)
    DeviceArray<uint32_t> d_kbits;    // [B][H][WW] NMS survivors of the fused edge kernel
    DeviceArray<uint8_t> d_vplane;    // [B][H][W]  their magnitudes (sparse: only survivors' bytes are ever written / read)
    DeviceArray<int> d_pre;           // [B] magnitude floor per frame | [B] floor of the redo pass | [B] redo list | count
    DeviceArray<uint32_t> d_roi_bits;     // [n_roi][roi_stride] bit-planes of the ROI masks, each [H][WW]
    int n_roi = 0;                        // ROI masks; with more than one, frame f uses mask stream_id[f]
    size_t roi_stride = 0;                // words between ROI planes: H*WW rounded up to 128 bytes (bulk-copy sources)
    DeviceArray<int> d_roi_idx;           // [2][B] ROI plane of each frame, per result slot (n_roi > 1 only)
    DeviceArray<uint32_t> d_pmask_bits;   // [B][bh][WW] ROI-masked edges (the HoughLinesP mask)
    DeviceArray<uint32_t> d_edge_bits;    // [B][H][WW] Canny map
    DeviceArray<uint32_t> d_cand_bits, d_strong_bits;   // [B][H][WW] candidate / strong planes before hysteresis
    // generic-width fallback (byte maps), allocated on first use
    DeviceArray<uint8_t> d_cls, d_cls_dbg, d_roi, d_pmask;   // d_roi: [n_roi][H*W]
    std::vector<uint8_t> h_roi;                               // [n_roi][H*W]
    bool fallback_ready = false, last_cluster = false;
    int last_paths = 0;               // LANE_PATH_* of the chunk that ran last
    DeviceArray<uint8_t> d_gray_dbg;
    DeviceArray<uint32_t> d_hist, d_points, d_points_dbg;
    DeviceArray<uint8_t> d_lut;       // low[511] | high[511]
    DeviceArray<int4> d_thr;
    DeviceArray<int> d_seedsA, d_seedsB, d_seed_count;
    int seed_cap = 0;
    DeviceArray<int> d_n_edges, d_n_points, d_rounds, d_n_lines;
    DeviceArray<int32_t> d_lines;
    DeviceArray<uint32_t> d_accum16;  // [B][cells_per_frame] biased 16-bit cells, two per word
    DeviceArray<int2> d_win;          // [180] (rmin, first cell) per angle
    int cells_per_frame = 0;
    int ppht_v2 = 0;                  // LANE_B200_K4=v2 pins the global-memory PPHT kernel (tests)
    DeviceArray<int> d_order;         // [B] frames with the most points first (v3 launch order)
    DeviceArray<int2> d_win3;         // v3 layout: (rmin, first cell inside the owning CTA)
    DeviceArray<uint32_t> d_pmask_work;   // [B][G3][bh][WW] private mask copies of the v3 cluster CTAs
    DeviceArray<uint32_t> d_list_over;    // [B][G3][over_cap] private extensions of the v3 point list (ROIs with many pixels)
    int G3 = 0, cells_max3 = 0, list_cap3 = 0, over_cap3 = 0;   // v3 plan: cluster size, cells / shared list entries per CTA, list extension
    DeviceArray<double> d_fit_raw, d_fit_big;             // LaneFitScratch
    DeviceArray<int> d_fit_side_n, d_fit_side_flags;
    DeviceArray<int> d_stream_id;
    DeviceArray<double> d_prev_fit;
    DeviceArray<uint8_t> d_prev_valid;
    int stream_cap = 0;
    DeviceArray<int32_t> d_std_accum;
    // batched standard Hough (lane_hough_lines_batch), allocated on first use
    DeviceArray<int32_t> d_hb_accum, d_hb_sorted;
    DeviceArray<int2> d_hb_tmp;
    DeviceArray<int> d_hb_count;
    CudaEvent hb_ev[2];
    DeviceArray<int2> d_peaks;
    DeviceArray<int> d_n_peaks;
    DeviceArray<int> d_task_counter;

    // Up to two batches may be in flight on the context's stream (enqueue, enqueue, collect, enqueue, collect ...): the
    // device never waits for the host between them.  Each has its own pinned result buffers and timing events.
    struct slot_t {
        PinnedArray<lane_record> h_records;
        DeviceArray<lane_record> d_records;          // alive until this slot is enqueued again
        PinnedArray<double> h_prev_fit;              // state in (explicit mode) and state out
        PinnedArray<uint8_t> h_prev_valid;
        PinnedArray<int32_t> h_roi_idx;              // staging of d_roi_idx (n_roi > 1 only)
        PinnedArray<RigFrame> h_rig;                 // staging of the slot's d_rig rows (lazy)
        // lane_rig_enqueue's host ticks: the slot's frames, copied whole while the other slot's tick computes (lazy,
        // grows), and the event after the ingest launch that last read them
        DeviceArray<uint8_t> d_src;
        CudaEvent src_read;
        CudaEvent ev[LANE_NUM_STAGES + 1];
        CudaEvent done;
        CudaEvent reader_done;                       // lane_ctx_fence_records: an outside reader of d_records ends here
        bool has_reader = false;
        int n = 0, S = 0;
        bool timed = false;
        int32_t launches[LANE_NUM_STAGES] = {};
    } slots[2];
    int last_collected = 0;                          // slot of the batch lane_detect_collect returned last
    int q_first = 0, q_count = 0, cur = 0;           // oldest batch in flight, batches in flight, slot being / last enqueued
    bool state_on_device = false;                    // a batch has run: the EMA state of its streams is in d_prev_*
    const uint8_t *last_frames_dev = nullptr;
    float stage_ms[LANE_NUM_STAGES] = {};            // of the batch collected last
    int32_t stage_launches[LANE_NUM_STAGES] = {};

    // Waits for all work on the context's streams: what they may still read or write can then be released.
    cudaError_t sync() const
    {
        cudaError_t e = cudaStreamSynchronize(st);
        if (!e && st2) e = cudaStreamSynchronize(st2);
        if (!e && copy_st) e = cudaStreamSynchronize(copy_st);
        return e;
    }
    ~lane_ctx()                                      // the members release their resources after this
    {
        cudaSetDevice(device);
        sync();
    }
};

namespace {

int fail(lane_ctx *c, int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (c) c->err = buf; else g_create_error = buf;
    return code;
}

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(c, LANE_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                        __FILE__, __LINE__);                                                       \
    } while (0)

int ensure_streams(lane_ctx *c, int S)
{
    if (S <= c->stream_cap) return LANE_OK;
    CU(c->d_prev_fit.grow((size_t)S * 6));
    CU(c->d_prev_valid.grow((size_t)S * 2));
    for (auto &sl : c->slots) {
        CU(sl.h_prev_fit.alloc((size_t)S * 6));
        CU(sl.h_prev_valid.alloc((size_t)S * 2));
    }
    c->state_on_device = false;
    c->stream_cap = S;
    return LANE_OK;
}

// Staging `src` (the context's d_src or a slot's) for `need` bytes of host source frames.  A larger need replaces the
// buffer once the context's streams are idle (an earlier batch may still be copying into it or converting out of it).
int ensure_src(lane_ctx *c, DeviceArray<uint8_t> &src, size_t need)
{
    if (src && need > src.size()) CU(c->sync());
    CU(src.grow(need));
    return LANE_OK;
}

// Byte-map buffers of the generic-width path, allocated the first time that path runs.
int ensure_fallback(lane_ctx *c)
{
    if (c->fallback_ready) return LANE_OK;
    const size_t P = (size_t)c->g.H * c->g.W, B = (size_t)c->max_batch;
    CU(c->d_cls.alloc(B * P));
    if (c->debug) CU(c->d_cls_dbg.alloc(B * P));
    CU(c->d_roi.alloc(P * c->n_roi));
    CU(c->d_pmask.alloc(B * std::max(c->g.bw * c->g.bh, 1)));
    CU(c->d_seedsA.alloc(B * c->seed_cap));
    CU(c->d_seedsB.alloc(B * c->seed_cap));
    CU(c->d_seed_count.alloc(B));
    CU(cudaMemcpyAsync(c->d_roi, c->h_roi.data(), P * c->n_roi, cudaMemcpyHostToDevice, c->st));
    c->fallback_ready = true;
    return LANE_OK;
}

// LANE_B200_SYNC_DEBUG=1: synchronise after every stage and name the one that faulted (debugging aid)
int stage_check(lane_ctx *c, const char *what)
{
    static const bool on = getenv("LANE_B200_SYNC_DEBUG") != nullptr;
    if (!on) return LANE_OK;
    cudaError_t e = cudaStreamSynchronize(c->st);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) return fail(c, LANE_ERR_CUDA, "stage %s failed: %s", what, cudaGetErrorString(e));
    return LANE_OK;
}

int mark(lane_ctx *c, int i)
{
    if (c->profiling) CU(cudaEventRecord(c->slots[c->cur].ev[i], c->st));
    return LANE_OK;
}

// All pixel stages for frames [off, off+m) of the batch (per-frame buffers are indexed by the batch position).
int run_stages(lane_ctx *c, const uint8_t *frames_dev, int off, int m, const int32_t *stream_id_dev, int S, bool timed)
{
    const LaneGeom &g = c->g;
    const int H = g.H, W = g.W;
    const size_t P = (size_t)H * W, WW = (W + 31) / 32, planes = (size_t)H * WW, o = (size_t)off;
    int *L = c->slots[c->cur].launches;
    int rc;
    const uint8_t *fr = frames_dev + o * P * 3;
    uint32_t *hist = c->d_hist + o * 256;
    // what the edge half hands to the back half lives in the batch's result slot: the edge kernels of the next batch may
    // already be writing while PPHT / fit of this one still read
    const size_t two = o + (size_t)c->cur * c->max_batch;
    int4 *thr = c->d_thr + two;
    int *n_edges = c->d_n_edges + two, *n_points = c->d_n_points + two, *rounds = c->d_rounds + two, *n_lines = c->d_n_lines + o;
    uint32_t *points = c->d_points + two * g.max_points;
    uint32_t *pmask_bits = c->d_pmask_bits + two * std::max(g.bh, 1) * WW;
    uint32_t *edge_bits = c->d_edge_bits + o * planes, *cb = c->d_cand_bits + o * planes, *sb = c->d_strong_bits + o * planes;
    int32_t *lines = c->d_lines + o * g.max_segments * 4;
    // ROI plane per frame: null (plane 0 for every frame) on a single-ROI context
    const int *roi_idx = c->n_roi > 1 ? c->d_roi_idx + two : nullptr;
    const size_t roi_stride = roi_idx ? c->roi_stride : 0;

    if (timed) { rc = mark(c, LANE_STAGE_BLUR_HIST); if (rc) return rc; }
    // Fused edge path (aligned widths, Gaussian blur on): one kernel from BGR frames to NMS survivors, then the
    // cluster kernel; the blurred plane is only written for the verification taps.
    bool fused = false;
    c->last_cluster = false;
    if (c->blur && lane_fused_edge_supported(H, W, fr)) {
        CU(c->d_kbits.lazy((size_t)c->max_batch * planes));
        CU(c->d_vplane.lazy((size_t)c->max_batch * P));
        CU(c->d_pre.lazy((size_t)c->max_batch * 5 + 4));
        if (c->debug) CU(c->d_blur.lazy((size_t)c->max_batch * P));
        const size_t B = (size_t)c->max_batch;
        int *pre = c->d_pre + o, *pre_redo = c->d_pre + B + o, *redo_list = c->d_pre + 2 * B + o, *redo_flag = c->d_pre + 3 * B + o,
            *frame_done = c->d_pre + 4 * B + o, *redo_count = c->d_pre + 5 * B;
        uint32_t *kb = c->d_kbits + o * planes;
        uint8_t *vp = c->d_vplane + o * P, *bd = c->debug ? c->d_blur + o * P : nullptr;
        int *LK = &L[LANE_STAGE_BLUR_HIST], *LC = &L[LANE_STAGE_CANNY];
        if (launch_fused_edge(fr, c->d_lut, c->d_lut + 511, hist, thr, pre, pre_redo, redo_list, redo_count, redo_flag, frame_done,
                              kb, vp, bd, c->d_task_counter, m, H, W, c->st, LK)) {
            rc = stage_check(c, "k1_fused"); if (rc) return rc;
            if (timed) { rc = mark(c, LANE_STAGE_CANNY); if (rc) return rc; }
            fused = launch_canny_cluster_fused(kb, vp, hist, c->d_lut, c->d_lut + 511, c->d_roi_bits, roi_idx, roi_stride, thr,
                                               pre, pre_redo, redo_list, redo_count, redo_flag, nullptr, n_edges, rounds, points, n_points,
                                               pmask_bits, edge_bits, cb, sb, g, m, c->st, LC) &&
                    // frames whose sampled floor was above their true low (normally none): rebuild K / V with the exact
                    // floor and finish them; both kernels return at once when the list is empty
                    launch_fused_edge_redo(fr, redo_list, redo_count, pre_redo, kb, vp, bd, c->d_task_counter, m, H, W, c->st, LC) &&
                    launch_canny_cluster_fused(kb, vp, hist, c->d_lut, c->d_lut + 511, c->d_roi_bits, roi_idx, roi_stride, thr,
                                               pre, pre_redo, redo_list, redo_count, redo_flag, redo_list, n_edges, rounds, points, n_points,
                                               pmask_bits, edge_bits, cb, sb, g, m, c->st, LC);
        }
        if (!fused) fprintf(stderr, "lane_b200: fused edge path rejected by device %d, using the unfused kernels\n", c->device);
        c->last_cluster = fused;
        rc = stage_check(c, "k2_canny_cluster (fused input)"); if (rc) return rc;
        if (getenv("LANE_B200_SYNC_DEBUG")) {
            int nredo = 0;
            cudaMemcpy(&nredo, redo_count, sizeof(int), cudaMemcpyDeviceToHost);
            if (nredo) fprintf(stderr, "lane_b200: %d of %d frames redone with the exact magnitude floor\n", nredo, m);
        }
    }
    c->last_paths = fused ? LANE_PATH_FUSED_EDGE : 0;
    if (!fused) {
        CU(c->d_blur.lazy((size_t)c->max_batch * P));
        uint8_t *blur = c->d_blur + o * P;
        if (timed) { rc = mark(c, LANE_STAGE_BLUR_HIST); if (rc) return rc; }
        launch_blur_hist(fr, blur, hist, m, H, W, c->st, &L[LANE_STAGE_BLUR_HIST], c->blur);
        if (timed) { rc = mark(c, LANE_STAGE_CANNY); if (rc) return rc; }
        c->last_cluster =
            launch_canny_cluster(blur, hist, c->d_lut, c->d_lut + 511, c->d_roi_bits, roi_idx, roi_stride, thr, n_edges, rounds,
                                 points, n_points,
                                 pmask_bits, edge_bits, cb, sb, c->d_task_counter, g, m, c->st, &L[LANE_STAGE_CANNY]);
    }
    if (c->last_cluster) {
        if (timed) { rc = mark(c, LANE_STAGE_COMPACT); if (rc) return rc; }
    } else {
        // generic widths / unaligned planes: byte-map kernels, then the same bit-plane outputs
        rc = ensure_fallback(c); if (rc) return rc;
        uint8_t *cls = c->d_cls + o * P, *blur = c->d_blur + o * P;
        int *seedsA = c->d_seedsA + o * c->seed_cap, *seedsB = c->d_seedsB + o * c->seed_cap, *seed_count = c->d_seed_count + o;
        launch_thresholds(hist, c->d_lut, c->d_lut + 511, thr, m, H, W, c->st, &L[LANE_STAGE_CANNY]);
        launch_sobel_nms(blur, thr, cls, seedsA, seed_count, c->seed_cap, m, H, W, c->st, &L[LANE_STAGE_CANNY]);
        if (c->debug) CU(cudaMemcpyAsync(c->d_cls_dbg + o * P, cls, (size_t)m * P, cudaMemcpyDeviceToDevice, c->st));
        launch_hysteresis(cls, seedsA, seedsB, seed_count, c->seed_cap, rounds, m, H, W, c->st, &L[LANE_STAGE_CANNY]);
        launch_finalize_edges(cls, n_edges, m, H, W, c->st, &L[LANE_STAGE_CANNY]);
        if (timed) { rc = mark(c, LANE_STAGE_COMPACT); if (rc) return rc; }
        launch_compact(cls, c->d_roi, roi_idx, roi_idx ? P : 0, c->d_pmask + o * std::max(g.bw * g.bh, 1), points, n_points,
                       g, m, c->st, &L[LANE_STAGE_COMPACT]);
        launch_bytes_to_bits(cls, edge_bits, m, H, W, W, c->st, &L[LANE_STAGE_COMPACT]);
        launch_mask_rows(edge_bits, c->d_roi_bits, roi_idx, roi_stride, pmask_bits, g, m, c->st, &L[LANE_STAGE_COMPACT]);
    }
    c->last_paths |= c->last_cluster ? LANE_PATH_CLUSTER_CANNY : 0;
    if (c->debug)
        CU(cudaMemcpyAsync(c->d_points_dbg + o * g.max_points, points, sizeof(uint32_t) * (size_t)m * g.max_points,
                           cudaMemcpyDeviceToDevice, c->st));

    rc = stage_check(c, "canny / compaction"); if (rc) return rc;
    if (timed) { rc = mark(c, LANE_STAGE_PPHT); if (rc) return rc; }
    cudaStream_t hs = c->st;                       // stream of the back half
    if (c->overlap_now) {
        hs = c->st2;
        CU(cudaEventRecord(c->edge_done[c->cur], c->st));
        CU(cudaStreamWaitEvent(hs, c->edge_done[c->cur], 0));
    }
    // v3 (cells in distributed shared memory) takes every frame it can; v2 (global 16-bit cells) then sweeps
    // up the frames v3 flagged (point list larger than its shared-memory list), or runs alone if v3 cannot launch.
    bool v3 = !c->ppht_v2 && c->G3 > 0 &&
              launch_ppht_v3(points, n_points, pmask_bits, c->d_pmask_work + o * c->G3 * std::max(g.bh, 1) * WW,
                             c->d_list_over ? c->d_list_over + o * c->G3 * (size_t)c->over_cap3 : nullptr, c->d_win3, c->cells_max3, c->list_cap3, c->over_cap3, c->G3, lines, n_lines, g, c->hp, m, hs, &L[LANE_STAGE_PPHT],
                             c->d_order + o);
    launch_ppht_v2(points, n_points, pmask_bits, c->d_accum16 + o * (c->cells_per_frame / 2), c->d_win,
                   c->cells_per_frame, lines, n_lines, g, c->hp, m, hs, &L[LANE_STAGE_PPHT], v3 ? 1 : 0);
    if (v3) c->last_paths |= LANE_PATH_PPHT_DSMEM;

    rc = stage_check(c, "ppht"); if (rc) return rc;
    if (timed) { rc = mark(c, LANE_STAGE_FIT); if (rc) return rc; }
    if (c->slots[c->cur].has_reader) {             // an outside reader (the NCCL gather) may still be on this slot's records
        CU(cudaStreamWaitEvent(hs, c->slots[c->cur].reader_done, 0));
        c->slots[c->cur].has_reader = false;
    }
    LaneFitScratch fs{c->d_fit_raw + o * 6, c->d_fit_side_n + o * 2, c->d_fit_side_flags + o,
                      c->d_fit_big ? c->d_fit_big + o * 2 * 5 * 2 * (size_t)g.max_segments : nullptr};
    launch_fit(lines, n_lines, fs, stream_id_dev ? stream_id_dev + o : nullptr, S, c->d_prev_fit, c->d_prev_valid, c->smooth,
               c->one_minus_smooth, thr, n_edges, n_points, rounds, c->slots[c->cur].d_records + o, g, m, hs, &L[LANE_STAGE_FIT]);
    return stage_check(c, "fit");
}

// What a batch enqueues before its frames: the stream its back half runs on, its stream ids, every frame's ROI plane
// and, when given, the explicit EMA state it starts from.
int begin_batch(lane_ctx *c, bool on_device, int n, const int32_t *stream_id, int S, const double *prev_fit,
                const uint8_t *prev_valid)
{
    lane_ctx::slot_t &sl = c->slots[c->cur];
    // back half on its own stream: device-resident batches outside profiling / debug mode (stage events and taps assume
    // one stream).  Everything only the back half touches (stream ids, EMA state, records) is ordered on that stream.
    const bool was_overlap = c->overlap_now;
    c->overlap_now = on_device && !c->profiling && !c->debug;
    if (was_overlap != c->overlap_now && c->q_count) {       // mode change with a batch in flight: order the two streams once
        CU(cudaEventRecord(c->edge_done[c->cur ^ 1], was_overlap ? c->st2 : c->st));
        CU(cudaStreamWaitEvent(was_overlap ? c->st : c->st2, c->edge_done[c->cur ^ 1], 0));
    }
    cudaStream_t hs = c->overlap_now ? c->st2 : c->st;
    if (stream_id) CU(cudaMemcpyAsync(c->d_stream_id, stream_id, sizeof(int) * n, cudaMemcpyHostToDevice, hs));
    if (c->n_roi > 1) {
        // The edge kernels read each frame's ROI plane from their own copy of the stream ids, made on the compute stream:
        // d_stream_id is written on the back half's stream while the fit of the batch before may still read it.
        if (stream_id) memcpy(sl.h_roi_idx, stream_id, sizeof(int32_t) * n);
        else memset(sl.h_roi_idx, 0, sizeof(int32_t) * n);
        CU(cudaMemcpyAsync(c->d_roi_idx + (size_t)c->cur * c->max_batch, sl.h_roi_idx, sizeof(int32_t) * n,
                           cudaMemcpyHostToDevice, c->st));
    }
    if (prev_fit) {                                  // explicit state: the caller's; otherwise what the last batch left on the device
        memcpy(sl.h_prev_fit, prev_fit, sizeof(double) * S * 6);
        memcpy(sl.h_prev_valid, prev_valid, (size_t)S * 2);
        CU(cudaMemcpyAsync(c->d_prev_fit, sl.h_prev_fit, sizeof(double) * S * 6, cudaMemcpyHostToDevice, hs));
        CU(cudaMemcpyAsync(c->d_prev_valid, sl.h_prev_valid, (size_t)S * 2, cudaMemcpyHostToDevice, hs));
    }
    return LANE_OK;
}

// Host frames are cut into chunks that are copied on a second stream while the previous chunk computes (the EMA state
// stays on the device across chunks, which run in order on the compute stream).  Chunks of this many frames let a copy
// (~50 GB/s) and the compute of the previous chunk overlap; >= 4 chunks when possible.
int host_chunk(int n) { return std::max(1, std::min(64, (n + 3) / 4)); }

// The copy stream of host batches (created on first use), and where a batch's copies start: once the work enqueued
// before them is done with the staging they write.  That is everything on the compute stream, or for a batch staged
// in its result slot only the ingest launch that last read the slot's staging: its copies then run under the batch
// in flight.
int begin_host_copies(lane_ctx *c, bool staged)
{
    if (!c->copy_st) {
        for (auto &e : c->copy_ev) CU(e.create(cudaEventDisableTiming));
        CU(c->start_ev.create(cudaEventDisableTiming));
        for (auto &sl : c->slots) CU(sl.src_read.create(cudaEventDisableTiming));
        CU(c->copy_st.create(cudaStreamNonBlocking));
    }
    if (staged) {
        CU(cudaStreamWaitEvent(c->copy_st, c->slots[c->cur].src_read, 0));
    } else {
        CU(cudaEventRecord(c->start_ev, c->st));
        CU(cudaStreamWaitEvent(c->copy_st, c->start_ev, 0));
    }
    return LANE_OK;
}

// The compute stream waits for the copies of chunk k.
int chunk_copied(lane_ctx *c, int k)
{
    cudaEvent_t ev = c->copy_ev[k % LANE_COPY_EVENTS];
    CU(cudaEventRecord(ev, c->copy_st));
    CU(cudaStreamWaitEvent(c->st, ev, 0));
    return LANE_OK;
}

// What a batch enqueues after its frames: the copies of its records and of the EMA state after it, and its entry in the
// queue of batches in flight.
int end_batch(lane_ctx *c, bool on_device, int n, int S, const uint8_t *frames_dev)
{
    lane_ctx::slot_t &sl = c->slots[c->cur];
    cudaStream_t hs = c->overlap_now ? c->st2 : c->st;
    int rc = mark(c, LANE_STAGE_D2H); if (rc) return rc;
    CU(cudaMemcpyAsync(sl.h_records, sl.d_records, sizeof(lane_record) * n, cudaMemcpyDeviceToHost, hs));
    CU(cudaMemcpyAsync(sl.h_prev_fit, c->d_prev_fit, sizeof(double) * S * 6, cudaMemcpyDeviceToHost, hs));
    CU(cudaMemcpyAsync(sl.h_prev_valid, c->d_prev_valid, (size_t)S * 2, cudaMemcpyDeviceToHost, hs));
    rc = mark(c, LANE_NUM_STAGES); if (rc) return rc;
    CU(cudaGetLastError());
    c->last_frames_dev = frames_dev;
    CU(cudaEventRecord(sl.done, hs));
    sl.n = n;
    sl.S = S;
    sl.timed = c->profiling && on_device;
    c->state_on_device = true;
    c->q_count++;
    return LANE_OK;
}

// How the context's H x W BGR frames are made from the batch's sources before the path runs (k0_common.cuh): they
// already are those frames; one launch_ingest over frames of one layout and size; or k0_rig_ingest over every frame,
// each with its own layout and size, driven by the batch's descriptor table.
enum class Ingest { none, single, rig };

// Enqueue a validated batch: the frames of `sources` in source order, all on the device or all in host memory.  Device
// frames are read where they are.  Host frames land one after another in a device buffer, behind the compute of what
// came before.  Host frames `staged` (lane_rig_enqueue, page-locked) are copied whole into the result slot's own
// staging, after the ingest that last read it; the batch then runs like a device batch.  Other host frames are copied
// chunk by chunk (host_chunk) into the context's buffers, each chunk behind the compute of the chunk before.
int enqueue(lane_ctx *c, const lane_rig_source *sources, int n_sources, bool on_device, bool staged, Ingest ingest,
            int n, const int32_t *stream_id, int S, const double *prev_fit, const uint8_t *prev_valid)
{
    staged = staged && !on_device;
    const bool whole = on_device || staged;          // one chunk: one ingest launch and one pass of the path
    lane_ctx::slot_t &sl = c->slots[c->cur];
    const size_t B = (size_t)c->max_batch, bgr_bytes = (size_t)c->g.H * c->g.W * 3;
    if (ingest != Ingest::none || !on_device) CU(c->d_frames.lazy(B * bgr_bytes));
    // host frame f lands at byte offset at[f]: in the context's frames when they need no ingest, else in source staging
    std::vector<size_t> at(n + 1, 0);
    for (int s = 0, f = 0; s < n_sources; s++) {
        const lane_rig_source &r = sources[s];
        for (int j = 0; j < r.n; j++, f++) at[f + 1] = at[f] + lane_input_frame_bytes(r.format, r.src_h, r.src_w);
    }
    uint8_t *land = c->d_frames;
    if (!on_device && ingest != Ingest::none) {
        DeviceArray<uint8_t> &src = staged ? sl.d_src : c->d_src;
        const int rc = ensure_src(c, src, at[n]);
        if (rc) return rc;
        land = src;
    }
    if (ingest == Ingest::rig) {
        CU(c->d_rig.lazy(2 * B));
        if (!sl.h_rig) CU(sl.h_rig.alloc(B));
        for (int s = 0, f = 0; s < n_sources; s++) {
            const lane_rig_source &r = sources[s];
            if (!r.n) continue;
            RigFrame d;
            CU(rig_frame(nullptr, r.format, r.src_h, r.src_w, c->g.H, c->g.W, &d));
            for (int j = 0; j < r.n; j++, f++) {
                d.src = on_device ? r.frames + j * lane_input_frame_bytes(r.format, r.src_h, r.src_w) : land + at[f];
                sl.h_rig[f] = d;
            }
        }
    }
    int rc = begin_batch(c, whole, n, stream_id, S, prev_fit, prev_valid);
    if (rc) return rc;
    RigFrame *rig = ingest == Ingest::rig ? c->d_rig + (size_t)c->cur * B : nullptr;
    if (rig) CU(cudaMemcpyAsync(rig, sl.h_rig, sizeof(RigFrame) * n, cudaMemcpyHostToDevice, c->st));
    const int32_t *sid = stream_id ? c->d_stream_id.get() : nullptr;
    const uint8_t *frames_dev = on_device && ingest == Ingest::none ? sources[0].frames : c->d_frames.get();
    // pinned (or registered) host frames go straight to the copy engine, ordinary memory through the device's staging
    // ring when the batch is large; decided once per source for the whole batch
    std::vector<HostStager *> ring(n_sources, nullptr);
    if (!on_device) {
        for (int s = 0; s < n_sources; s++)
            if (sources[s].n && HostStager::pageable(sources[s].frames, at[n])) ring[s] = &lane_device_host(c->device).stager;
        rc = begin_host_copies(c, staged); if (rc) return rc;
    }
    const int chunk = whole ? n : host_chunk(n);
    for (int off = 0, k = 0; off < n; off += chunk, k++) {
        const int m = std::min(chunk, n - off);
        if (!on_device) {
            // the chunk's frames of each source are contiguous on both sides: one copy per source
            for (int s = 0, first = 0; s < n_sources && first < off + m; first += sources[s].n, s++) {
                const int lo = std::max(off, first), hi = std::min(off + m, first + sources[s].n);
                if (lo >= hi) continue;
                const lane_rig_source &r = sources[s];
                const uint8_t *from = r.frames + (lo - first) * lane_input_frame_bytes(r.format, r.src_h, r.src_w);
                if (ring[s])
                    CU(ring[s]->h2d(land + at[lo], from, at[hi] - at[lo], c->copy_st));
                else
                    CU(cudaMemcpyAsync(land + at[lo], from, at[hi] - at[lo], cudaMemcpyHostToDevice, c->copy_st));
            }
            rc = chunk_copied(c, staged ? c->cur : k); if (rc) return rc;
        }
        uint8_t *to = c->d_frames + (size_t)off * bgr_bytes;
        if (ingest == Ingest::single) {                // one source: its frames are contiguous on either side
            const lane_rig_source &r = sources[0];
            CU(launch_ingest((on_device ? r.frames : land) + at[off], r.format, m, r.src_h, r.src_w, to, c->g.H, c->g.W, c->st));
        } else if (rig) {
            launch_rig_ingest(rig + off, m, to, c->g.H, c->g.W, c->st);
        }
        if (staged) CU(cudaEventRecord(sl.src_read, c->st));
        rc = run_stages(c, frames_dev, off, m, sid, S, whole && c->profiling);
        if (rc) return rc;
    }
    return end_batch(c, whole, n, S, frames_dev);
}

// One source's fields: layout and size (lane_input_refusal) and frames.  `s` numbers it in the message; < 0: the call's
// only source.
int check_source(lane_ctx *c, int s, const lane_rig_source &r)
{
    char who[32] = "";
    if (s >= 0) snprintf(who, sizeof(who), "source %d: ", s);
    if (r.src_h < 1 || r.src_w < 1) return fail(c, LANE_ERR_INVALID, "%sbad source size %dx%d", who, r.src_w, r.src_h);
    if (const char *why = lane_input_refusal(r.format, r.src_h, r.src_w))
        return fail(c, LANE_ERR_INVALID, "%s%s (format %d, %dx%d)", who, why, r.format, r.src_w, r.src_h);
    if (r.n && !r.frames) return fail(c, LANE_ERR_INVALID, "%sframes is null", who);
    return LANE_OK;
}

// The ingest kernels that resize put the batch's frames on the grid's z.
int check_grid(lane_ctx *c, long long n)
{
    return n > 65535 ? fail(c, LANE_ERR_UNSUPPORTED, "batch %lld above 65535", n) : LANE_OK;
}

// The checks lane_detect_rig and lane_rig_enqueue share before check_call: every source's fields, the batch size, and
// the stream id of every frame (into `stream_id`).  Returns the batch's frame count or a LANE_ERR_* code.
int check_rig(lane_ctx *c, const lane_rig_source *sources, int n_sources, int n_streams, std::vector<int32_t> &stream_id)
{
    long long n = 0;
    for (int s = 0; s < n_sources; s++) {
        const lane_rig_source &r = sources[s];
        if (r.n < 0) return fail(c, LANE_ERR_INVALID, "source %d: negative frame count %d", s, r.n);
        if (const int rc = check_source(c, s, r)) return rc;
        if (r.stream_id < 0 || r.stream_id >= n_streams)
            return fail(c, LANE_ERR_INVALID, "source %d: stream_id %d outside [0,%d)", s, r.stream_id, n_streams);
        n += r.n;
    }
    if (n < 1 || n > c->max_batch) return fail(c, LANE_ERR_INVALID, "bad batch: %lld frames (max_batch=%d)", n, c->max_batch);
    if (const int rc = check_grid(c, n)) return rc;
    for (int s = 0; s < n_sources; s++) stream_id.insert(stream_id.end(), sources[s].n, sources[s].stream_id);
    return (int)n;
}

// Whether host memory [p, p + bytes) is page-locked or registered, so the copy engine reads it where it is.
bool page_locked(const void *p, size_t bytes)
{
    return host_memory_type(p) == cudaMemoryTypeHost && host_memory_type((const uint8_t *)p + bytes - 1) == cudaMemoryTypeHost;
}

// What every detect call checks and sets up before it enqueues: arguments and context state, the context's device, the
// stream state buffers, the batch's result slot and, when profiling, the mark where the batch starts.
int check_call(lane_ctx *c, const void *frames, int n, const int32_t *stream_id, int S, const void *pf, const void *pv)
{
    if (!c) return LANE_ERR_INVALID;
    if (!frames || n <= 0 || n > c->max_batch) return fail(c, LANE_ERR_INVALID, "bad batch: n=%d (max_batch=%d)", n, c->max_batch);
    if (S <= 0 || (!pf) != (!pv)) return fail(c, LANE_ERR_INVALID, "bad stream state: n_streams=%d", S);
    if (!c->have_roi || !c->have_lut) return fail(c, LANE_ERR_STATE, "lane_set_roi_mask and lane_set_threshold_lut must be called first");
    if (c->n_roi > 1 && S > c->n_roi)
        return fail(c, LANE_ERR_INVALID, "n_streams=%d but the context holds %d ROI masks (one per stream)", S, c->n_roi);
    if (pf) {          // explicit state is staged through host buffers: one batch at a time
        if (c->q_count) return fail(c, LANE_ERR_STATE, "a batch is already in flight; call lane_detect_collect");
    } else {           // state carried on the device: a second batch may queue behind the first
        if (c->q_count >= 2) return fail(c, LANE_ERR_STATE, "two batches are already in flight; call lane_detect_collect");
        if (!c->state_on_device || S > c->stream_cap)
            return fail(c, LANE_ERR_STATE, "no state on the device for %d streams: pass prev_fit / prev_valid once", S);
    }
    if (stream_id)
        for (int i = 0; i < n; i++)
            if (stream_id[i] < 0 || stream_id[i] >= S)
                return fail(c, LANE_ERR_INVALID, "stream_id[%d]=%d outside [0,%d)", i, stream_id[i], S);
    CU(cudaSetDevice(c->device));
    if (!c->q_count) {
        const int rc = ensure_streams(c, S);
        if (rc) return rc;
    }
    c->cur = (c->q_first + c->q_count) & 1;
    memset(c->slots[c->cur].launches, 0, sizeof(c->slots[c->cur].launches));
    if (c->profiling) CU(cudaEventRecord(c->slots[c->cur].ev[LANE_STAGE_H2D], c->st));
    return LANE_OK;
}

// Enqueue the frames of a single-format call (checked by check_call) as a batch of one source, with the caller's
// stream id per frame.  They need an ingest unless they are BGR at the context's size.
int enqueue_frames(lane_ctx *c, const lane_rig_source &r, bool on_device, const int32_t *stream_id, int S,
                   const double *prev_fit, const uint8_t *prev_valid)
{
    const bool resizes = lane_input_resizes(r.format, r.src_h, r.src_w, c->g.H, c->g.W);
    if (resizes)
        if (const int rc = check_grid(c, r.n)) return rc;
    const Ingest ingest = r.format == LANE_INPUT_BGR && !resizes ? Ingest::none : Ingest::single;
    return enqueue(c, &r, 1, on_device, false, ingest, r.n, stream_id, S, prev_fit, prev_valid);
}

// lane_detect_batch and its ingest forms: validate, enqueue, collect.
int detect_blocking(lane_ctx *c, const lane_rig_source &r, bool on_device, const int32_t *stream_id, int n_streams,
                    double *prev_fit, uint8_t *prev_valid, lane_record *out)
{
    int rc = check_source(c, -1, r);
    if (rc) return rc;
    rc = check_call(c, r.frames, r.n, stream_id, n_streams, prev_fit, prev_valid);
    if (rc) return rc;
    if (!out) return fail(c, LANE_ERR_INVALID, "out is null");
    rc = enqueue_frames(c, r, on_device, stream_id, n_streams, prev_fit, prev_valid);
    if (rc) return rc;
    return lane_detect_collect(c, prev_fit, prev_valid, out);
}

// The queries on the last batch (taps, Hough, edge counts) need it collected and, when they name one of its frames,
// that frame to exist; otherwise it must hold a frame at all.  Returns the batch's size or a LANE_ERR_* code.
int last_batch(lane_ctx *c, const int *frame_index = nullptr)
{
    if (c->q_count) return fail(c, LANE_ERR_STATE, "collect the last batch first");
    const int n = c->slots[c->cur].n;
    if (frame_index && (*frame_index < 0 || *frame_index >= n))
        return fail(c, LANE_ERR_INVALID, "frame_index %d outside the last batch (%d frames)", *frame_index, n);
    if (n < 1) return fail(c, LANE_ERR_STATE, "no batch has run on this context");
    return n;
}

// Words of one ROI bit-plane: [H][WW], padded to 128 bytes so that every plane's rows are aligned bulk-copy sources.
size_t roi_plane_words(const LaneGeom &g) { return ((size_t)g.H * ((g.W + 31) / 32) + 31) & ~(size_t)31; }

// The streams, events and buffers a context has from its creation on; the rest are created on first use.
int create_resources(lane_ctx *c)
{
    const size_t B = (size_t)c->max_batch, H = (size_t)c->g.H, WW = (c->g.W + 31) / 32;
    CU(c->st.create(cudaStreamNonBlocking));
    {
        // the back half first: its clusters keep their slots, the edge kernels fill in (DESIGN.md §4, "Two streams")
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        CU(c->st2.create(cudaStreamNonBlocking, hi));
        for (auto &e : c->edge_done) CU(e.create(cudaEventDisableTiming));
    }
    for (auto &sl : c->slots) {
        for (auto &e : sl.ev) CU(e.create());
        CU(sl.done.create(cudaEventDisableTiming));
        CU(sl.reader_done.create(cudaEventDisableTiming));
    }
    CU(c->d_roi_bits.alloc(roi_plane_words(c->g)));           // one plane; more are made by lane_set_roi_masks
    CU(c->d_edge_bits.alloc(B * H * WW));
    CU(c->d_cand_bits.alloc(B * H * WW));
    CU(c->d_strong_bits.alloc(B * H * WW));
    CU(c->d_hist.alloc(B * 256));
    CU(c->d_lut.alloc(1022));
    CU(c->d_thr.alloc(2 * B));
    CU(c->d_n_edges.alloc(2 * B));
    CU(c->d_n_points.alloc(2 * B));
    CU(c->d_rounds.alloc(2 * B));
    CU(c->d_n_lines.alloc(B));
    CU(c->d_order.alloc(B));
    CU(c->d_win.alloc(LANE_NUM_ANGLES));
    CU(c->d_win3.alloc(LANE_NUM_ANGLES));
    CU(c->d_lines.alloc(B * c->g.max_segments * 4));
    CU(c->d_fit_raw.alloc(B * 6));
    CU(c->d_fit_side_n.alloc(B * 2));
    CU(c->d_fit_side_flags.alloc(B));
    if (c->g.max_segments > LANE_MAX_SIDE_SEGMENTS)      // a side can hold every segment: work columns in global memory
        CU(c->d_fit_big.alloc(B * 2 * 5 * 2 * (size_t)c->g.max_segments));
    CU(c->d_stream_id.alloc(B));
    for (auto &sl : c->slots) {
        CU(sl.d_records.alloc(B));
        CU(cudaMemset(sl.d_records, 0, sizeof(lane_record) * B));
    }
    CU(c->d_task_counter.alloc(4));
    for (auto &sl : c->slots) CU(sl.h_records.alloc(B));
    lane_upload_tables();
    CU(cudaGetLastError());
    CU(cudaDeviceSynchronize());
    return LANE_OK;
}

}  // namespace

extern "C" {

int lane_abi_version(void) { return LANE_B200_ABI_VERSION; }

const char *lane_last_error(const lane_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int lane_ctx_create(int device, int height, int width, int max_batch, int max_segments, lane_ctx **out)
{
    lane_ctx *c = nullptr;   // errors before allocation go to the global slot
    if (!out) return fail(c, LANE_ERR_INVALID, "out is null");
    *out = nullptr;
    if (height < 1 || width < 1 || max_batch < 1) return fail(c, LANE_ERR_INVALID, "bad shape %dx%d batch %d", height, width, max_batch);
    if (height > 32767 || width > 32767) return fail(c, LANE_ERR_UNSUPPORTED, "frame %dx%d exceeds 32767 px per side", height, width);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(c, LANE_ERR_NO_DEVICE, "no CUDA device visible: this library has no CPU fallback");
    if (device < 0 || device >= std::min(ndev, LANE_MAX_DEVICES))
        return fail(c, LANE_ERR_INVALID, "device %d out of range (%d visible)", device, ndev);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major != 10)
        return fail(c, LANE_ERR_NO_DEVICE, "device %d is sm_%d%d; this build holds sm_100a code only", device, prop.major, prop.minor);
    if (cudaSetDevice(device) != cudaSuccess) return fail(c, LANE_ERR_CUDA, "cudaSetDevice(%d) failed", device);

    auto ctx = std::make_unique<lane_ctx>();
    ctx->device = device;
    ctx->max_batch = max_batch;
    LaneGeom &g = ctx->g;
    g.H = height; g.W = width;
    g.numrho = 2 * (width + height) + 1;
    g.max_segments = max_segments > 0 ? max_segments : 256;
    ctx->seed_cap = (int)std::min<size_t>((size_t)height * width, (size_t)1 << 17);
    {
        const char *e = getenv("LANE_B200_K4");
        ctx->ppht_v2 = e && !strcmp(e, "v2");
    }
    if (const int rc = create_resources(ctx.get())) {
        g_create_error = std::move(ctx->err);        // the context goes; lane_last_error(NULL) reads why
        cudaGetLastError();                          // reported: not left behind for the next call's own check
        return rc;
    }
    *out = ctx.release();
    return LANE_OK;
}

void lane_ctx_destroy(lane_ctx *ctx) { delete ctx; }

int lane_set_roi_mask(lane_ctx *c, const uint8_t *mask) { return lane_set_roi_masks(c, mask, 1); }

int lane_set_roi_masks(lane_ctx *c, const uint8_t *masks, int n_masks)
{
    if (!c || !masks || n_masks < 1) return LANE_ERR_INVALID;
    CU(cudaSetDevice(c->device));
    // Detect calls are refused until every buffer made from the ROI is rebuilt below, so a re-set that fails part way
    // leaves a context without a ROI, not one whose kernels would read released buffers.  The old buffers go before the
    // new ones are allocated: the two sets are never held at once.
    c->have_roi = false;
    CU(c->sync());
    c->fallback_ready = false;                       // the generic-width buffers are rebuilt on next use
    c->d_cls.reset(); c->d_cls_dbg.reset(); c->d_roi.reset(); c->d_pmask.reset();
    c->d_seedsA.reset(); c->d_seedsB.reset(); c->d_seed_count.reset();
    c->d_pmask_bits.reset(); c->d_points.reset(); c->d_points_dbg.reset();
    c->d_accum16.reset(); c->d_pmask_work.reset(); c->d_list_over.reset();
    c->d_roi_idx.reset();
    for (auto &sl : c->slots) sl.h_roi_idx.reset();
    if (n_masks > 1) c->d_roi_bits.reset();         // one plane stays where lane_ctx_create put it

    // Every buffer and window made from the ROI below comes from the union of the masks: a frame's point list and
    // HoughLinesP mask hold only its own mask's pixels, and rows or rho windows beyond its own mask's reach stay empty.
    // The point lists are sized by the largest mask.
    LaneGeom &g = c->g;
    const size_t P = (size_t)g.H * g.W, WW = (g.W + 31) / 32;
    const size_t stride = roi_plane_words(g);
    std::vector<uint8_t> uni(masks, masks + P);
    std::vector<uint32_t> bits(stride * n_masks, 0u);
    int x0 = g.W, y0 = g.H, x1 = -1, y1 = -1, cnt = 0;
    for (int r = 0; r < n_masks; r++) {
        const uint8_t *mask = masks + r * P;
        uint32_t *plane = bits.data() + r * stride;
        int mask_cnt = 0;
        for (int y = 0; y < g.H; y++)
            for (int x = 0; x < g.W; x++)
                if (mask[(size_t)y * g.W + x]) {
                    x0 = std::min(x0, x); x1 = std::max(x1, x); y0 = std::min(y0, y); y1 = std::max(y1, y);
                    mask_cnt++;
                    uni[(size_t)y * g.W + x] = 1;
                    plane[(size_t)y * WW + (x >> 5)] |= 1u << (x & 31);
                }
        cnt = std::max(cnt, mask_cnt);
    }
    if (x1 < 0) { x0 = y0 = 0; x1 = y1 = -1; }
    g.bx0 = x0; g.by0 = y0; g.bx1 = x1 + 1; g.by1 = y1 + 1;
    g.bw = g.bx1 - g.bx0; g.bh = g.by1 - g.by0;
    g.max_points = cnt;
    c->n_roi = n_masks;
    c->roi_stride = stride;
    c->h_roi.assign(masks, masks + P * n_masks);
    CU(c->d_roi_bits.grow(bits.size()));
    CU(cudaMemcpy(c->d_roi_bits, bits.data(), sizeof(uint32_t) * bits.size(), cudaMemcpyHostToDevice));
    if (n_masks > 1) {
        CU(c->d_roi_idx.alloc(2 * (size_t)c->max_batch));
        CU(cudaMemset(c->d_roi_idx, 0, sizeof(int) * 2 * (size_t)c->max_batch));   // valid planes for taps of an older batch
        for (auto &sl : c->slots) CU(sl.h_roi_idx.alloc((size_t)c->max_batch));
    }
    {
        int2 win[LANE_NUM_ANGLES];
        c->cells_per_frame = lane_ppht_windows(uni.data(), g.H, g.W, win);
        CU(cudaMemcpy(c->d_win, win, sizeof(win), cudaMemcpyHostToDevice));
        CU(c->d_accum16.alloc((size_t)c->max_batch * (c->cells_per_frame / 2)));
        int2 win3[LANE_NUM_ANGLES];
        c->G3 = lane_ppht_plan_v3(win, c->cells_per_frame, win3, &c->cells_max3, &c->list_cap3);
        {
            // v3 keeps a frame's cells in the shared memory of a cluster, so the number of frames in flight is what the
            // cells leave room for: 74 at 1080p (G = 4, two CTAs per SM) but only 18 at 4K (G = 16), where the
            // global-memory kernel with every frame of the batch in flight is faster (measured on B200, 128 x 4K:
            // v3 3.55 ms, v2 2.47 ms).  Take v3 only when it can keep at least 32 frames going.
            if (c->G3 > 0) {
                const size_t per_cta = (size_t)c->cells_max3 * 2 + sizeof(uint32_t) * (size_t)c->list_cap3 + 4700;
                const int ctas = per_cta <= 112 * 1024 ? 2 : 1;
                if (lane_sm_count() * ctas / c->G3 < 32) c->G3 = 0;
            }
        }
        CU(cudaMemcpy(c->d_win3, win3, sizeof(win3), cudaMemcpyHostToDevice));
        if (c->G3 > 0) {
            CU(c->d_pmask_work.alloc((size_t)c->max_batch * c->G3 * std::max(g.bh, 1) * WW));
            // the ROI can hold more edge pixels than the shared-memory list: every CTA of a cluster gets a private global
            // extension, sized by the ROI up to lane_ppht_over_cap_v3() points (busier frames go to the global-memory kernel)
            c->over_cap3 = 0;
            if (cnt > c->list_cap3) {
                c->over_cap3 = (int)std::min<long long>((long long)cnt - c->list_cap3, lane_ppht_over_cap_v3());
                c->over_cap3 = (c->over_cap3 + 63) & ~63;
                CU(c->d_list_over.alloc((size_t)c->max_batch * c->G3 * (size_t)c->over_cap3));
            }
        }
    }
    CU(c->d_pmask_bits.alloc(2 * (size_t)c->max_batch * std::max(g.bh, 1) * WW));      // per result slot
    CU(c->d_points.alloc(2 * (size_t)c->max_batch * g.max_points));
    if (c->debug) CU(c->d_points_dbg.alloc((size_t)c->max_batch * g.max_points));
    c->have_roi = true;
    return LANE_OK;
}

int lane_set_threshold_lut(lane_ctx *c, const uint8_t *low511, const uint8_t *high511)
{
    if (!c || !low511 || !high511) return LANE_ERR_INVALID;
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->st));
    CU(cudaMemcpy(c->d_lut, low511, 511, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(c->d_lut + 511, high511, 511, cudaMemcpyHostToDevice));
    c->have_lut = true;
    return LANE_OK;
}

int lane_set_hough_params(lane_ctx *c, int threshold, int min_line_length, int max_line_gap)
{
    if (!c || threshold < 1 || min_line_length < 0 || max_line_gap < 0) return LANE_ERR_INVALID;
    c->hp = LaneHoughParams{threshold, min_line_length, max_line_gap};
    return LANE_OK;
}

int lane_set_smoothing(lane_ctx *c, double factor, double one_minus_factor)
{
    if (!c) return LANE_ERR_INVALID;
    c->smooth = factor; c->one_minus_smooth = one_minus_factor;
    return LANE_OK;
}

int lane_set_preprocess(lane_ctx *c, int gaussian_blur)
{
    if (!c) return LANE_ERR_INVALID;
    c->blur = gaussian_blur != 0;
    return LANE_OK;
}

int lane_set_debug(lane_ctx *c, int keep)
{
    if (!c) return LANE_ERR_INVALID;
    CU(cudaSetDevice(c->device));
    c->debug = keep != 0;
    if (c->debug) {
        const size_t P = (size_t)c->g.H * c->g.W;
        if (c->fallback_ready) CU(c->d_cls_dbg.lazy((size_t)c->max_batch * P));
        CU(c->d_gray_dbg.lazy(P));
        if (c->have_roi) CU(c->d_points_dbg.lazy((size_t)c->max_batch * c->g.max_points));
    }
    return LANE_OK;
}

int lane_set_profiling(lane_ctx *c, int enabled)
{
    if (!c) return LANE_ERR_INVALID;
    c->profiling = enabled != 0;
    return LANE_OK;
}

void *lane_ctx_stream(lane_ctx *c) { return c ? (void *)c->st : nullptr; }

int lane_ctx_last_paths(lane_ctx *c) { return c ? c->last_paths : 0; }

const lane_record *lane_ctx_records_device(lane_ctx *c) { return c ? c->slots[c->last_collected].d_records.get() : nullptr; }

int lane_ctx_fence_records(lane_ctx *c, void *reader_stream)
{
    if (!c) return LANE_ERR_INVALID;
    CU(cudaSetDevice(c->device));
    lane_ctx::slot_t &sl = c->slots[c->last_collected];
    CU(cudaEventRecord(sl.reader_done, (cudaStream_t)reader_stream));
    sl.has_reader = true;
    return LANE_OK;
}

int lane_ctx_set_stream(lane_ctx *c, void *cuda_stream)
{
    if (!c) return LANE_ERR_INVALID;
    if (c->q_count) return fail(c, LANE_ERR_STATE, "cannot switch streams with a batch in flight");
    if (c->st) cudaStreamSynchronize(c->st);
    c->st.borrow((cudaStream_t)cuda_stream);
    return LANE_OK;
}

int lane_detect_enqueue(lane_ctx *c, const uint8_t *frames_dev, int n, const int32_t *stream_id, int n_streams,
                        const double *prev_fit, const uint8_t *prev_valid)
{
    const int rc = check_call(c, frames_dev, n, stream_id, n_streams, prev_fit, prev_valid);
    if (rc) return rc;
    return enqueue_frames(c, {frames_dev, LANE_INPUT_BGR, c->g.H, c->g.W, n, 0}, true, stream_id, n_streams, prev_fit, prev_valid);
}

int lane_detect_collect(lane_ctx *c, double *prev_fit, uint8_t *prev_valid, lane_record *out)
{
    if (!c || !out || !prev_fit || !prev_valid) return LANE_ERR_INVALID;
    if (!c->q_count) return fail(c, LANE_ERR_STATE, "no batch in flight");
    CU(cudaSetDevice(c->device));
    lane_ctx::slot_t &sl = c->slots[c->q_first];     // the oldest batch; a younger one keeps running
    c->last_collected = c->q_first;
    c->q_first ^= 1;
    c->q_count--;
    CU(cudaEventSynchronize(sl.done));
    memcpy(out, sl.h_records, sizeof(lane_record) * sl.n);
    memcpy(prev_fit, sl.h_prev_fit, sizeof(double) * sl.S * 6);
    memcpy(prev_valid, sl.h_prev_valid, (size_t)sl.S * 2);
    memcpy(c->stage_launches, sl.launches, sizeof(c->stage_launches));
    if (sl.timed)
        for (int i = 0; i < LANE_NUM_STAGES; i++) CU(cudaEventElapsedTime(&c->stage_ms[i], sl.ev[i], sl.ev[i + 1]));
    return LANE_OK;
}

int lane_detect_batch(lane_ctx *c, const uint8_t *frames, int frames_on_device, int n, const int32_t *stream_id,
                      int n_streams, double *prev_fit, uint8_t *prev_valid, lane_record *out)
{
    if (!c) return LANE_ERR_INVALID;
    return detect_blocking(c, {frames, LANE_INPUT_BGR, c->g.H, c->g.W, n, 0}, frames_on_device != 0, stream_id, n_streams,
                           prev_fit, prev_valid, out);
}

int lane_detect_batch_nv12(lane_ctx *c, const uint8_t *frames_nv12, int frames_on_device, int n, const int32_t *stream_id,
                           int n_streams, double *prev_fit, uint8_t *prev_valid, lane_record *out)
{
    if (!c) return LANE_ERR_INVALID;
    return detect_blocking(c, {frames_nv12, LANE_INPUT_NV12, c->g.H, c->g.W, n, 0}, frames_on_device != 0, stream_id,
                           n_streams, prev_fit, prev_valid, out);
}

int lane_detect_batch_ingest(lane_ctx *c, const uint8_t *frames, int frames_on_device, int n, int format, int src_h,
                             int src_w, const int32_t *stream_id, int n_streams, double *prev_fit, uint8_t *prev_valid,
                             lane_record *out)
{
    if (!c) return LANE_ERR_INVALID;
    return detect_blocking(c, {frames, format, src_h, src_w, n, 0}, frames_on_device != 0, stream_id, n_streams, prev_fit,
                           prev_valid, out);
}

int lane_detect_rig(lane_ctx *c, const lane_rig_source *sources, int n_sources, int frames_on_device, int n_streams,
                    double *prev_fit, uint8_t *prev_valid, lane_record *out)
{
    if (!c || !sources || !out || !prev_fit || !prev_valid)
        return fail(c, LANE_ERR_INVALID, "lane_detect_rig: ctx, sources, prev_fit, prev_valid and out must not be null");
    std::vector<int32_t> stream_id;
    const int n = check_rig(c, sources, n_sources, n_streams, stream_id);
    if (n < 0) return n;
    int rc = check_call(c, sources, n, stream_id.data(), n_streams, prev_fit, prev_valid);
    if (rc) return rc;
    rc = enqueue(c, sources, n_sources, frames_on_device != 0, false, Ingest::rig, n, stream_id.data(), n_streams, prev_fit,
                 prev_valid);
    if (rc) return rc;
    return lane_detect_collect(c, prev_fit, prev_valid, out);
}

int lane_rig_enqueue(lane_ctx *c, const lane_rig_source *sources, int n_sources, int frames_on_device, int n_streams,
                     const double *prev_fit, const uint8_t *prev_valid)
{
    if (!c || !sources) return fail(c, LANE_ERR_INVALID, "lane_rig_enqueue: ctx and sources must not be null");
    std::vector<int32_t> stream_id;
    const int n = check_rig(c, sources, n_sources, n_streams, stream_id);
    if (n < 0) return n;
    if (!frames_on_device)
        for (int s = 0; s < n_sources; s++)
            if (const lane_rig_source &r = sources[s];
                r.n && !page_locked(r.frames, lane_input_frame_bytes(r.format, r.src_h, r.src_w, r.n)))
                return fail(c, LANE_ERR_INVALID, "source %d: host frames must be page-locked or registered memory "
                            "(cudaHostAlloc, cudaHostRegister, torch pin_memory)", s);
    const int rc = check_call(c, sources, n, stream_id.data(), n_streams, prev_fit, prev_valid);
    if (rc) return rc;
    return enqueue(c, sources, n_sources, frames_on_device != 0, true, Ingest::rig, n, stream_id.data(), n_streams, prev_fit,
                   prev_valid);
}

int lane_get_stage_ms(lane_ctx *c, float ms[LANE_NUM_STAGES], int32_t launches[LANE_NUM_STAGES])
{
    if (!c) return LANE_ERR_INVALID;
    if (ms) memcpy(ms, c->stage_ms, sizeof(c->stage_ms));
    if (launches) memcpy(launches, c->stage_launches, sizeof(c->stage_launches));
    return LANE_OK;
}

int lane_debug_tap(lane_ctx *c, int what, int fi, void *host_out, size_t capacity, size_t *bytes_written)
{
    if (!c || !host_out) return LANE_ERR_INVALID;
    if (const int n = last_batch(c, &fi); n < 0) return n;
    CU(cudaSetDevice(c->device));
    const LaneGeom &g = c->g;
    const size_t P = (size_t)g.H * g.W;
    const void *src = nullptr;
    size_t bytes = 0;
    std::vector<int32_t> tmp;
    switch (what) {
    case LANE_TAP_BLUR:
        if (!c->d_blur) return fail(c, LANE_ERR_STATE, "LANE_TAP_BLUR needs lane_set_debug(ctx,1) before detect");
        src = c->d_blur + fi * P; bytes = P; break;
    case LANE_TAP_HIST: src = c->d_hist + fi * 256; bytes = 256 * sizeof(uint32_t); break;
    case LANE_TAP_EDGES:
    case LANE_TAP_CLASS: {
        const size_t WW = (g.W + 31) / 32, words = (size_t)g.H * WW;
        if (P > capacity) return fail(c, LANE_ERR_INVALID, "tap needs %zu bytes, capacity %zu", P, capacity);
        uint8_t *o = (uint8_t *)host_out;
        if (what == LANE_TAP_EDGES) {
            std::vector<uint32_t> e(words);
            CU(cudaMemcpy(e.data(), c->d_edge_bits + fi * words, sizeof(uint32_t) * words, cudaMemcpyDeviceToHost));
            for (int y = 0; y < g.H; y++)
                for (int x = 0; x < g.W; x++)
                    o[(size_t)y * g.W + x] = ((e[y * WW + (x >> 5)] >> (x & 31)) & 1u) ? 255 : 0;
        } else if (!c->debug) {
            return fail(c, LANE_ERR_STATE, "LANE_TAP_CLASS needs lane_set_debug(ctx,1) before detect");
        } else if (c->last_cluster) {
            std::vector<uint32_t> cc(words), ss(words);
            CU(cudaMemcpy(cc.data(), c->d_cand_bits + fi * words, sizeof(uint32_t) * words, cudaMemcpyDeviceToHost));
            CU(cudaMemcpy(ss.data(), c->d_strong_bits + fi * words, sizeof(uint32_t) * words, cudaMemcpyDeviceToHost));
            for (int y = 0; y < g.H; y++)
                for (int x = 0; x < g.W; x++) {
                    const uint32_t cb = (cc[y * WW + (x >> 5)] >> (x & 31)) & 1u, sb = (ss[y * WW + (x >> 5)] >> (x & 31)) & 1u;
                    o[(size_t)y * g.W + x] = (uint8_t)(sb ? 2 : cb);
                }
        } else {
            CU(cudaMemcpy(o, c->d_cls_dbg + fi * P, P, cudaMemcpyDeviceToHost));
        }
        if (bytes_written) *bytes_written = P;
        return LANE_OK;
    }
    case LANE_TAP_GRAY:
        if (!c->d_gray_dbg) return fail(c, LANE_ERR_STATE, "LANE_TAP_GRAY needs lane_set_debug(ctx,1)");
        launch_gray_debug(c->last_frames_dev + fi * P * 3, c->d_gray_dbg, g.H, g.W, c->st);
        CU(cudaStreamSynchronize(c->st));
        src = c->d_gray_dbg; bytes = P; break;
    case LANE_TAP_POINTS: {
        if (!c->debug || !c->d_points_dbg) return fail(c, LANE_ERR_STATE, "LANE_TAP_POINTS needs lane_set_debug(ctx,1) before detect");
        int np = c->slots[c->cur].h_records[fi].n_roi_points;
        std::vector<uint32_t> packed(np);
        CU(cudaMemcpy(packed.data(), c->d_points_dbg + (size_t)fi * g.max_points, sizeof(uint32_t) * np, cudaMemcpyDeviceToHost));
        bytes = sizeof(int32_t) * 2 * np;
        if (bytes > capacity) return fail(c, LANE_ERR_INVALID, "tap needs %zu bytes, capacity %zu", bytes, capacity);
        int32_t *o = (int32_t *)host_out;
        for (int i = 0; i < np; i++) { o[2 * i] = packed[i] & 0xFFFF; o[2 * i + 1] = packed[i] >> 16; }
        if (bytes_written) *bytes_written = bytes;
        return LANE_OK;
    }
    case LANE_TAP_FRAME: src = c->last_frames_dev + fi * P * 3; bytes = P * 3; break;
    case LANE_TAP_SEGMENTS:
        src = c->d_lines + (size_t)fi * g.max_segments * 4;
        bytes = sizeof(int32_t) * 4 * c->slots[c->cur].h_records[fi].n_segments; break;
    default: return fail(c, LANE_ERR_INVALID, "unknown tap %d", what);
    }
    if (bytes > capacity) return fail(c, LANE_ERR_INVALID, "tap needs %zu bytes, capacity %zu", bytes, capacity);
    if (bytes) CU(cudaMemcpy(host_out, src, bytes, cudaMemcpyDeviceToHost));
    if (bytes_written) *bytes_written = bytes;
    return LANE_OK;
}

int lane_hough_accumulator(lane_ctx *c, int fi, int32_t *accum_host, int threshold, int32_t *peaks_host,
                           int max_peaks, int *n_peaks)
{
    if (!c) return LANE_ERR_INVALID;
    if (const int n = last_batch(c, &fi); n < 0) return n;
    if (!c->debug || !c->d_points_dbg) return fail(c, LANE_ERR_STATE, "lane_hough_accumulator needs lane_set_debug(ctx,1) before detect");
    CU(cudaSetDevice(c->device));
    const LaneGeom &g = c->g;
    const size_t cells = (size_t)(LANE_NUM_ANGLES + 2) * (g.numrho + 2);
    CU(c->d_std_accum.lazy(cells));
    launch_hough_accum(c->d_points_dbg + (size_t)fi * g.max_points, c->d_n_points + (size_t)c->cur * c->max_batch + fi, c->d_std_accum, g, c->st);
    CU(cudaGetLastError());
    if (accum_host) CU(cudaMemcpyAsync(accum_host, c->d_std_accum, sizeof(int32_t) * cells, cudaMemcpyDeviceToHost, c->st));
    int found = 0;
    if (peaks_host && max_peaks > 0) {
        CU(c->d_peaks.grow((size_t)max_peaks));
        CU(c->d_n_peaks.lazy(1));
        launch_hough_peaks(c->d_std_accum, g.numrho, threshold, c->d_peaks, max_peaks, c->d_n_peaks, c->st);
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync(&found, c->d_n_peaks, sizeof(int), cudaMemcpyDeviceToHost, c->st));
        CU(cudaStreamSynchronize(c->st));
        int m = std::min(found, max_peaks);
        std::vector<int2> pk(m);
        CU(cudaMemcpy(pk.data(), c->d_peaks, sizeof(int2) * m, cudaMemcpyDeviceToHost));
        // cv2 order: votes descending, flat index ascending
        std::sort(pk.begin(), pk.end(), [](const int2 &a, const int2 &b) { return a.y != b.y ? a.y > b.y : a.x < b.x; });
        for (int i = 0; i < m; i++) {
            int nn = pk[i].x / (g.numrho + 2) - 1;
            int r = pk[i].x - (nn + 1) * (g.numrho + 2) - 1;
            peaks_host[3 * i] = r; peaks_host[3 * i + 1] = nn; peaks_host[3 * i + 2] = pk[i].y;
        }
    }
    CU(cudaStreamSynchronize(c->st));
    if (n_peaks) *n_peaks = found;
    return LANE_OK;
}

int lane_edge_count_rect(lane_ctx *c, int x0, int y0, int x1, int y1, int32_t *counts_host)
{
    if (!c || !counts_host) return LANE_ERR_INVALID;
    const int n = last_batch(c);
    if (n < 0) return n;
    if (x0 < 0 || y0 < 0 || x1 > c->g.W || y1 > c->g.H || x0 >= x1 || y0 >= y1)
        return fail(c, LANE_ERR_INVALID, "bad rectangle [%d,%d) x [%d,%d)", x0, x1, y0, y1);
    CU(cudaSetDevice(c->device));
    // d_n_lines is free between batches (K5 has consumed it); reuse it as the result buffer
    launch_edge_count_rect(c->d_edge_bits, c->d_n_lines, n, c->g.H, c->g.W, x0, y0, x1, y1, c->st);
    CU(cudaMemcpyAsync(counts_host, c->d_n_lines, sizeof(int) * n, cudaMemcpyDeviceToHost, c->st));
    CU(cudaStreamSynchronize(c->st));
    CU(cudaGetLastError());
    return LANE_OK;
}

int lane_hough_lines_batch(lane_ctx *c, int threshold, int max_peaks, int32_t *peaks_host, int32_t *n_peaks_host,
                           int32_t *accum_host, float *device_ms)
{
    if (!c || max_peaks < 1 || !peaks_host || !n_peaks_host) return LANE_ERR_INVALID;
    const int n = last_batch(c);
    if (n < 0) return n;
    CU(cudaSetDevice(c->device));
    const LaneGeom &g = c->g;
    const size_t cells = (size_t)(LANE_NUM_ANGLES + 2) * (g.numrho + 2), B = (size_t)c->max_batch;
    CU(c->d_hb_sorted.grow(B * max_peaks * 3));
    CU(c->d_hb_tmp.grow(B * max_peaks));
    if (!c->d_hb_count) {
        for (auto &e : c->hb_ev) CU(e.create());
        CU(c->d_hb_count.alloc(B));
    }
    if (accum_host) CU(c->d_hb_accum.lazy(B * cells));
    CU(cudaEventRecord(c->hb_ev[0], c->st));
    const int *roi_idx = c->n_roi > 1 ? c->d_roi_idx + (size_t)c->cur * B : nullptr;
    if (!launch_hough_batch(c->d_edge_bits, c->d_roi_bits, roi_idx, roi_idx ? c->roi_stride : 0,
                            accum_host ? c->d_hb_accum.get() : nullptr, c->d_hb_tmp, c->d_hb_sorted, c->d_hb_count, g, threshold,
                            max_peaks, n, c->st))
        return fail(c, LANE_ERR_UNSUPPORTED, "frame %dx%d: a Hough row does not fit shared memory", g.W, g.H);
    CU(cudaEventRecord(c->hb_ev[1], c->st));
    CU(cudaMemcpyAsync(n_peaks_host, c->d_hb_count, sizeof(int) * n, cudaMemcpyDeviceToHost, c->st));
    CU(cudaMemcpyAsync(peaks_host, c->d_hb_sorted, sizeof(int32_t) * (size_t)n * max_peaks * 3, cudaMemcpyDeviceToHost, c->st));
    if (accum_host)
        CU(cudaMemcpyAsync(accum_host, c->d_hb_accum, sizeof(int32_t) * (size_t)n * cells, cudaMemcpyDeviceToHost, c->st));
    CU(cudaStreamSynchronize(c->st));
    CU(cudaGetLastError());
    if (device_ms) CU(cudaEventElapsedTime(device_ms, c->hb_ev[0], c->hb_ev[1]));
    return LANE_OK;
}

}  // extern "C"
