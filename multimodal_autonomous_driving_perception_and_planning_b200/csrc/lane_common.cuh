// Shared declarations for the lane-detection kernels (sm_100a).
//
// Stage map (reference lines are under /root/reference/src/perception/lane_detector.py):
//   K1  k1_blur_hist.cu   gray (:69) + 5x5 binomial blur (:72) + 256-bin histogram (:79)
//   K2  k2_cluster.cu     median/thresholds (:79-81) + Sobel + NMS (k2a), then hysteresis (:83) + ROI mask
//                         (:86-90) + row-major point list (HoughLinesP's nzloc) in one cluster per frame (k2b)
//       k2_canny.cu       byte-map fallback of the same stages for sizes the bit-plane path does not take
//   K3  k3_hough.cu       standard Hough accumulator + peaks (north-star add-on)
//   K4  k4_ppht.cu        exact cv2.HoughLinesP (:94-101)
//   K5  k5_fit.cu         side split (:105-134), polyfit + EMA + points (:136-176), offset (:253-272)
// Adjacent rows (SURVEY.md 8f):
//   K0  k0_resize.cu      cv2.resize of VideoDataLoader.read_frame (data/loaders/video_loader.py:108,128)
//       k0_nv12.cu        decoder output (NV12 / I420) -> BGR at the same size
//       k0_ingest.cu      decoder output -> BGR -> cv2.resize in one pass; the ingest launcher (k0_common.cuh)
//   K6  k6_frame_stats.cu mean / Laplacian variance / HSV green ratio of SceneClassifier (src/tagging/scene_classifier.py)
//   K7  k7_draw.cu        cv2-exact rasteriser: draw_lanes (:220-251), draw_lane_offset_indicator (visualization/overlays.py:103-148),
//                         the synthetic generator's frames (draw_prims.h: host expansion + the geometry shared with the device)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/lane_b200.h"

#define LANE_NUM_ANGLES 180
#define LANE_MAX_SIDE_SEGMENTS 256   // per side in shared memory; contexts with a larger max_segments use global scratch

struct LaneGeom {
    int H, W;
    int bx0, by0, bx1, by1;   // bounding box [bx0,bx1) x [by0,by1) of the ROI (of all ROI planes); empty => bx1 <= bx0
    int bw, bh;               // bbox size
    int numrho;               // 2*(W+H)+1
    int max_points;           // non-zero pixels of the largest ROI mask (upper bound of the point list)
    int max_segments;
};

struct LaneHoughParams {
    int threshold, min_len, max_gap;
};

// Function attributes (dynamic shared memory limit, non-portable cluster size) and the SM count are per DEVICE, and one
// process may drive several GPUs: "done once" flags are therefore arrays indexed by the current device.
#define LANE_MAX_DEVICES 64
static inline int lane_cur_device()
{
    int d = 0;
    cudaGetDevice(&d);
    return d & (LANE_MAX_DEVICES - 1);
}
static inline int lane_sm_count()
{
    static int sms[LANE_MAX_DEVICES];
    const int d = lane_cur_device();
    if (!sms[d]) cudaDeviceGetAttribute(&sms[d], cudaDevAttrMultiProcessorCount, d);
    return sms[d];
}

// message returned by lane_last_error(NULL): context creation and the context-free entry points
void lane_set_global_error(const char *msg);

// ---- K1 ---------------------------------------------------------------------------------
void launch_blur_hist(const uint8_t *frames, uint8_t *blur, uint32_t *hist, int n, int H, int W,
                      cudaStream_t st, int *launches, int gaussian_blur);
// fused edge kernel (k1_fused.cu): probe + gray + blur + histogram + Sobel + NMS -> K bit-plane, V byte plane
bool lane_fused_edge_supported(int H, int W, const void *frames);
bool launch_fused_edge(const uint8_t *frames, const uint8_t *lut_low, const uint8_t *lut_high, uint32_t *hist, int4 *thr,
                       int *pre, int *pre_redo, int *redo_list, int *redo_count, int *redo_flag, int *frame_done,
                       uint32_t *k_bits, uint8_t *v_plane, uint8_t *blur_dbg, int *task_counter, int n, int H, int W,
                       cudaStream_t st, int *launches);
bool launch_fused_edge_redo(const uint8_t *frames, const int *frame_list, const int *n_list, const int *pre,
                            uint32_t *k_bits, uint8_t *v_plane, uint8_t *blur_dbg, int *task_counter, int n, int H, int W,
                            cudaStream_t st, int *launches);
void launch_gray_debug(const uint8_t *frame, uint8_t *gray, int H, int W, cudaStream_t st);

// ---- K2 ---------------------------------------------------------------------------------
// thr: int4 per frame = (median_x2, low, high, 0)
void launch_thresholds(const uint32_t *hist, const uint8_t *lut_low, const uint8_t *lut_high, int4 *thr,
                       int n, int H, int W, cudaStream_t st, int *launches);
// cls: 0 none / 1 weak / 2 strong;  seeds: per-frame list of strong pixel indices
void launch_sobel_nms(const uint8_t *blur, const int4 *thr, uint8_t *cls, int *seeds, int *seed_count,
                      int seed_cap, int n, int H, int W, cudaStream_t st, int *launches);
// in place: promoted pixels become 3; afterwards cls >= 2 <=> edge.  rounds: per-frame BFS depth.
void launch_hysteresis(uint8_t *cls, int *seeds, int *seeds2, const int *seed_count, int seed_cap,
                       int *rounds, int n, int H, int W, cudaStream_t st, int *launches);
// cls (>=2) -> edges 0/255 in place, n_edges per frame
void launch_finalize_edges(uint8_t *cls_edges, int *n_edges, int n, int H, int W, cudaStream_t st, int *launches);
// ROI mask + ordered compaction: points[f][k] = (y<<16)|x in row-major order; pmask = bbox-sized byte mask.
// ROI planes (here and in every launcher below): frame f uses roi + roi_index[f] * roi_stride; a null roi_index means
// plane 0 for every frame.  The bounding box in g covers every plane.
void launch_compact(const uint8_t *edges, const uint8_t *roi, const int *roi_index, size_t roi_stride, uint8_t *pmask,
                    uint32_t *points, int *n_points, LaneGeom g, int n, cudaStream_t st, int *launches);

// cluster form of K2 (bit-planes in distributed shared memory); false => geometry not supported, use the kernels above
bool launch_canny_cluster(const uint8_t *blur, const uint32_t *hist, const uint8_t *lut_low, const uint8_t *lut_high,
                          const uint32_t *roi_bits, const int *roi_index, size_t roi_stride, int4 *thr, int *n_edges,
                          int *rounds, uint32_t *points,
                          int *n_points, uint32_t *pmask_bits, uint32_t *edge_bits, uint32_t *c_bits, uint32_t *s_bits,
                          int *task_counter, LaneGeom g, int n, cudaStream_t st, int *launches);
bool launch_canny_cluster_fused(const uint32_t *k_bits, const uint8_t *v_plane, const uint32_t *hist, const uint8_t *lut_low,
                                const uint8_t *lut_high, const uint32_t *roi_bits, const int *roi_index, size_t roi_stride,
                                int4 *thr, const int *pre, int *pre_redo, int *redo_list, int *redo_count, int *redo_flag,
                                const int *frame_list, int *n_edges, int *rounds, uint32_t *points, int *n_points,
                                uint32_t *pmask_bits, uint32_t *edge_bits, uint32_t *c_bits, uint32_t *s_bits, LaneGeom g, int n,
                                cudaStream_t st, int *launches);
void launch_edge_count_rect(const uint32_t *edge_bits, int *counts, int n, int H, int W, int x0, int y0, int x1, int y1,
                            cudaStream_t st);
void launch_bytes_to_bits(const uint8_t *bytes, uint32_t *bits, int n, int rows, int W, int row_stride,
                          cudaStream_t st, int *launches);
void launch_mask_rows(const uint32_t *edge_bits, const uint32_t *roi_bits, const int *roi_index, size_t roi_stride,
                      uint32_t *pmask_bits, LaneGeom g, int n, cudaStream_t st, int *launches);

// ---- K3 ---------------------------------------------------------------------------------
void launch_hough_accum(const uint32_t *points, const int *n_points, int32_t *accum_padded, LaneGeom g,
                        cudaStream_t st);
void launch_hough_peaks(const int32_t *accum_padded, int numrho, int threshold, int2 *peaks, int max_peaks,
                        int *n_peaks, cudaStream_t st);
// batched form: every frame of the batch, from the edge bit-planes (edge & ROI), peaks ordered on the device
bool launch_hough_batch(const uint32_t *edge_bits, const uint32_t *roi_bits, const int *roi_index, size_t roi_stride,
                        int32_t *accum, int2 *peaks_tmp, int32_t *peaks_sorted, int *n_peaks, LaneGeom g, int threshold,
                        int max_peaks, int n, cudaStream_t st);
void lane_upload_tables();       // trig tables -> __constant__ (both Hough variants)
void lane_upload_tables_std();

// ---- K4 ---------------------------------------------------------------------------------
// lines: int32 [n][max_segments][4]
// pmask_bits: [n][bh][WW] bit-plane of the ROI-masked edges (bit x&31 of word x>>5), cleared as lines are found
// v2: 16-bit biased cells inside per-angle rho windows (win[n] = (rmin, first cell)), producer warp, deep votes
void launch_ppht_v2(uint32_t *points, const int *n_points, uint32_t *pmask_bits, uint32_t *accum16, const int2 *win,
                    int cells_per_frame, int32_t *lines, int *n_lines, LaneGeom g, LaneHoughParams hp, int n,
                    cudaStream_t st, int *launches, int only_flagged);
int lane_ppht_windows(const uint8_t *mask, int H, int W, int2 *win);   // returns cells per frame
// v3: cells in distributed shared memory, cluster of G CTAs per frame, angle n owned by CTA n % G
int lane_ppht_plan_v3(const int2 *win, int cells_total, int2 *win3, int *cells_max, int *list_cap);
int lane_ppht_list_cap_v3();
int lane_ppht_over_cap_v3();
// list_over: [n][G][lane_ppht_over_cap_v3()] private list extensions (null = frames above the shared list go to v2)
bool launch_ppht_v3(const uint32_t *points, const int *n_points, const uint32_t *pmask_bits, uint32_t *pmask_work,
                    uint32_t *list_over, const int2 *win3, int cells_max, int list_cap, int over_cap, int G, int32_t *lines, int *n_lines, LaneGeom g,
                    LaneHoughParams hp, int n, cudaStream_t st, int *launches, int *order);

// ---- K5 ---------------------------------------------------------------------------------
struct LaneFitScratch {
    double *raw;        // [n][2][3]
    int *side_n;        // [n][2] segments per side (0 => None)
    int *side_flags;    // [n]
    double *big;        // [n][2][5][2 * max_segments] work columns when max_segments > LANE_MAX_SIDE_SEGMENTS, else null
};
void launch_fit(const int32_t *lines, const int *n_lines, LaneFitScratch fs, const int *stream_id, int n_streams,
                double *prev_fit, uint8_t *prev_valid, double smooth, double one_minus_smooth,
                const int4 *thr, const int *n_edges, const int *n_points, const int *rounds,
                lane_record *records, LaneGeom g, int n, cudaStream_t st, int *launches);

#ifdef __CUDACC__
// median of the blurred plane (x2) from its histogram; warp-collective
static __device__ __forceinline__ int median_x2_warp(const uint32_t *h, long long P, int lane)
{
    uint32_t c[8], s = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        c[i] = __ldcg(h + lane * 8 + i);   // from L2: the counts were accumulated with atomics by other SMs
        s += c[i];
    }
    uint32_t inc = s;
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    const long long exc = (long long)inc - s;
    const long long k0 = (P & 1) ? P / 2 : P / 2 - 1, k1 = P / 2;
    int v0 = -1, v1 = -1;
    long long run = exc;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        run += c[i];
        if (v0 < 0 && exc <= k0 && run > k0) v0 = lane * 8 + i;
        if (v1 < 0 && exc <= k1 && run > k1) v1 = lane * 8 + i;
    }
    for (int o = 16; o; o >>= 1) {
        v0 = max(v0, __shfl_xor_sync(0xffffffffu, v0, o));
        v1 = max(v1, __shfl_xor_sync(0xffffffffu, v1, o));
    }
    return v0 + v1;
}


// ---- TMA bulk copy (cp.async.bulk, SASS UBLKCP) + mbarrier helpers -------------------------------------
static __device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
static __device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
static __device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
static __device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
static __device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    asm volatile(
        "{\n\t.reg .pred p;\n"
        "W_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@!p bra W_%=;\n\t}"
        ::"r"(bar), "r"(parity) : "memory");
}
#endif
