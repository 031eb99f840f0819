// kernels.h — host-callable launchers of the CUDA kernels (one .cu per stage).
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

#include "common.cuh"
#include "p2p.cuh"

namespace stl {

// A keyframe on the banded three-kernel K1 (assoc2d_split.cu): an oversize keyframe (stl_allow_oversize_keyframes), or any
// keyframe under STL_K1_OVERSIZE=all.  Its slices of the three-kernel K1's workspace, which is indexed by oversize ordinal
// o (position in DevPack::ov) and laid out per candidate b as [b][n_ov] counters, [b][n_ov_kp] per-keypoint tables,
// [b][n_ov_surv] survivors and [b][n_ov_match] matches.
struct OvKf {
    int f;               // pack keyframe
    int surv_cap;        // survivor slots of one (candidate, keyframe) unit: max(kK1SurvCap, min(2 n_kp rounded up to 256, n_pad))
    int match_cap;       // match slots of one unit: 2 * surv_cap
    int n_bands;         // k_stream bands: ceil(bm_rows / k1_band_rows(bm_wpr))
    long long kp_off;    // first slot of its keypoints in [n_ov_kp]
    long long surv_off;  // first slot of its survivors in [n_ov_surv]
    long long match_off; // first slot of its matches in [n_ov_match]
};

// Device-resident pack (all pointers are device memory owned by the context).
struct DevPack {
    int n_kf = 0, n_covis = 0;
    long long n_pad_total = 0, n_nodes_total = 0, n_kp_total = 0, n_mp_total = 0;
    DevKf *kf = nullptr;
    float *px = nullptr, *py = nullptr, *pz = nullptr;
    uint32_t *orig = nullptr;
    float4 *node_lo = nullptr, *node_hi = nullptr;
    uint16_t *adj = nullptr;         // [n_nodes_total][32] leaf adjacency: the nearest leaves within adj_r of each leaf box (0xffff = none)
    float *adj_cov = nullptr;        // [n_nodes_total] squared distance the row covers (+inf: all of adj_r; -1: no row)
    PlaneRec *pl_rec = nullptr;      // [n_pad_total] plane index (null unless params.plane_index)
    int *pl_m = nullptr;             // [n_pad_total] neighbours kept; negative (-(m+1)) when the gates failed
    uint8_t *k1tab = nullptr;        // per-keyframe K1 table blobs (common.cuh: K1Tab), DevKf::tab_off / tab_bytes
    uint32_t *bitmap = nullptr;
    uint32_t *grid_start = nullptr;  // per keyframe gw*gh+1 entries
    uint32_t *grid_kp = nullptr;     // [n_kp_total] keypoint ids sorted by cell (local ids)
    float2 *kp_xy = nullptr;         // [n_kp_total]
    double2 *kp_xyd = nullptr;       // [n_kp_total] fp64 query pixels (variant 1 only; NaN = not queried)
    float *kp_mp = nullptr;          // [n_kp_total][3]
    float *Tcw = nullptr;            // [n_kf][12]
    float *relpose = nullptr;        // [n_kf][C][12]
    uint8_t *covis_valid = nullptr;  // [n_kf][C]
    float2 *covis_uv = nullptr;      // [n_kp_total][C]
    float *he_Tc = nullptr;          // [n_kf][12]
    double *he_Tl = nullptr;         // [n_kf][12]
    // keyframe selection (stl_select_keyframes): the kernels walk selection positions i < n_sel, keyframe sel_kf(pk, i), in
    // the order a pack of only those keyframes would have them.  sel == nullptr: every keyframe (n_sel = n_kf), no extra load.
    // Workspace records stay indexed by the pack's keyframe ([b][n_kf]): those of unselected keyframes are stale.
    int n_sel = 0;
    const int *sel = nullptr;        // [n_sel] selected keyframes, strictly increasing
    const int2 *sel_mp = nullptr;    // [n_sel + 1] (first compacted map-point slot of position i, mp_off - that): k_linearize's 3-D walk
    long long n_sel_mp = 0;          // map-point slots of the selected keyframes
    // three-kernel K1: the keyframes it serves (OvKf) and, for a launch, the ordinals of the selected ones, increasing
    int n_ov = 0;
    const OvKf *ov = nullptr;        // [n_ov]
    long long n_ov_kp = 0, n_ov_surv = 0, n_ov_match = 0;
    int n_ov_sel = 0;
    const int *ov_sel = nullptr;     // [n_ov_sel]
};

#ifdef __CUDACC__
__device__ __forceinline__ int sel_kf(const DevPack &pk, int i) { return pk.sel ? pk.sel[i] : i; }
#endif

// Workspace of one candidate chunk (Bc candidates x all keyframes).
struct DevWork {
    int Bc = 0;            // candidates per chunk
    int sub = 4;           // K2 sub-blocks per (candidate, keyframe)
    DevCand *cand = nullptr;      // [Bc]
    uint32_t *corr_kp = nullptr;  // [Bc][n_kp_total]  keypoint index of correspondence i of keyframe f at kp_off[f]+i
    uint32_t *corr_pt = nullptr;  // [Bc][n_kp_total]  original scan index
    uint32_t *corr_sp = nullptr;  // [Bc][n_kp_total]  sorted scan position
    uint32_t *q_corr = nullptr;   // [Bc][n_kp_total]  correspondence indices that carry a map point
    uint2 *q_kpsp = nullptr;      // [Bc][n_kp_total]  (keypoint, sorted scan position) of those, so that K2 needs no second hop
    int *n_corr = nullptr;        // [Bc][n_kf]
    int *n_q = nullptr;           // [Bc][n_kf]
    FrameRec *frame = nullptr;    // [Bc][n_kf]
    AlignRec *align = nullptr;    // [Bc][n_kf][sub]
    // neighbour lists of the 3-D queries, slot = b * n_mp_total + mp_off[f] + qi
    uint32_t *nn_pos = nullptr;   // [Bc][n_mp_total] sorted position of the 1-NN
    float *nn_g2 = nullptr;       // [Bc][n_mp_total] lower bound of the squared distance to any OTHER scan point (Sink1::g2)
    uint32_t *nb = nullptr;       // [Bc][n_mp_total][32] sorted positions of the k-NN, distance order
    float4 *nbx = nullptr;        // [32][Bc * n_mp_total] their coordinates, transposed (plane kernels read them coalesced)
    long long nbx_stride = 0;
    int *nb_m = nullptr;          // [Bc][n_mp_total] neighbours kept (d2 < radius^2)
    double *nb_last = nullptr;    // [Bc][n_mp_total] d2 of the last kept neighbour
    // optional per-query debug (allocated on demand, Bc_dbg = 1)
    uint32_t *dbg_nn = nullptr;   // [n_kp_total]
    int *dbg_m = nullptr;
    int *dbg_plane = nullptr;
    double *dbg_dist = nullptr;
    uint32_t *dbg_knn = nullptr;  // [n_kp_total][32]
    unsigned long long *dbg_stats = nullptr;  // [8] traversal statistics (debug runs)
    // K1 (assoc2d.cu) is persistent: k1_slots CTAs draw (candidate, keyframe) units from k1_ticket; the survivor records and
    // the match list are scratch of the CTA (slot = blockIdx.x), small enough to stay in L2
    int k1_slots = 0;
    int *k1_ticket = nullptr;        // [2] next chunk of units, CTAs that have left (the last one re-arms both)
    float4 *k1_rec = nullptr;        // [k1_slots][kK1SurvCap] (x, y, z, sorted position) of the points that passed the pre-cull
    ulonglong2 *k1_match = nullptr;  // [k1_slots][8192] matches of the exact pass
    // three-kernel K1 (assoc2d_split.cu), indexed by oversize ordinal (OvKf)
    ulonglong2 *k1_ov_match = nullptr;        // [Bc][n_ov_match] matches of the exact pass
    uint32_t *k1_surv = nullptr;              // [Bc][n_ov_surv] sorted positions that passed the pre-cull
    int *k1_cnt = nullptr;                    // [Bc][n_ov][4] survivors, matches, overflow flag, pad
    unsigned long long *k1_best_d2 = nullptr; // [Bc][n_ov_kp] bits of the smallest squared pixel distance per keypoint
    unsigned long long *k1_best_key = nullptr;// [Bc][n_ov_kp] (original index << 32 | position) of the point that owns it
    long long *k1_clk = nullptr;  // optional [units][8] phase clocks of K1 (diagnostic, STL_K1_CLK=1)
    int *overflow = nullptr;      // K1 survivor-list overflow counter (diagnostic)
};

// Device scratch of the index build, grown on demand and kept for the whole upload (a cudaMalloc / cudaFree
// pair per chunk of keyframes costs tens of milliseconds at these sizes).
struct BuildScratch {
    void *buf[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    size_t cap[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    cudaError_t need(int i, size_t bytes) {
        if (bytes <= cap[i]) return cudaSuccess;
        if (buf[i]) cudaFree(buf[i]);
        buf[i] = nullptr; cap[i] = 0;
        const cudaError_t e = cudaMalloc(&buf[i], bytes);
        if (e == cudaSuccess) cap[i] = bytes;
        return e;
    }
    void release() {
        for (int i = 0; i < 8; ++i) { if (buf[i]) cudaFree(buf[i]); buf[i] = nullptr; cap[i] = 0; }
    }
};

// ---- index build (build.cu) ---------------------------------------------------
// raw: [n][3] float32 device points of a chunk of keyframes; raw_off[nkf+1] host offsets.
// adj_r2: squared radius of the leaf adjacency lists (<= 0: none are built)
// kernel_ms (optional): the device time of the build kernels of this chunk is ADDED to it
cudaError_t build_scan_index(const float *d_raw, const long long *h_raw_off, int nkf, int kf_begin, const DevKf *h_kf,
                             DevPack &pack, float adj_r2, cudaStream_t st, BuildScratch &scr, float *kernel_ms = nullptr);

// plane index (knn3d.cu): k-NN + plane of every point of keyframes [kf_begin, kf_begin + nkf)
cudaError_t build_plane_index(const DevPack &pk, const DevKf *h_kf, int kf_begin, int nkf, const DevParams &pr, cudaStream_t st,
                              BuildScratch &scr);

constexpr int kK1SurvCap = 4096;   // survivors of the float32 pre-cull a (candidate, keyframe) unit may list
constexpr int kK1MatchCap = 8192;  // (keypoint, point) matches a unit may record between the exact pass and the tie pass
// Bands of the three-kernel K1's stream (DESIGN §3 "Oversize keyframes"): band j of a keyframe holds bitmap rows
// [j R, min((j + 1) R, bm_rows)) with R = k1_band_rows(bm_wpr), so that a band's words stay within kK1BandWords (16 KB)
// whatever the image size
constexpr int kK1BandWords = 4096;
__host__ __device__ inline int k1_band_rows(int bm_wpr) { return bm_wpr >= kK1BandWords ? 1 : kK1BandWords / bm_wpr; }

// ---- K1 (assoc2d.cu: one persistent kernel over the keyframes whose tables fit its shared memory; assoc2d_split.cu: banded
// stream / exact / correspondence kernels over the oversize keyframes DevPack::ov_sel) ----
size_t assoc2d_smem_bytes(int max_kp, int max_tab_bytes, int max_groups);
cudaError_t assoc2d_configure(size_t smem);
// with_terms = 0: correspondences only (the association pass of the LM path needs neither the covisible
// re-projection term nor the hand-eye term)
cudaError_t launch_assoc2d(const DevPack &pk, const DevWork &wk, const DevParams &pr, int B, size_t smem, int max_kp, int max_tab_bytes,
                           int max_groups, cudaStream_t st, int with_terms = 1);
// max_band_words: the largest band (rows * bm_wpr) of the served keyframes, at most kK1BandWords
size_t assoc2d_split_smem_bytes(int max_band_words, int max_groups);
cudaError_t assoc2d_split_configure(size_t smem);
// max_bands / max_surv_cap: maxima of OvKf::n_bands / surv_cap over DevPack::ov
cudaError_t launch_assoc2d_split(const DevPack &pk, const DevWork &wk, const DevParams &pr, int B, size_t smem, int max_bands, int max_surv_cap,
                                 cudaStream_t st, int with_terms = 1);

// ---- K2 (knn3d.cu) ---------------------------------------------------------------
// K2a (traversal: 1-NN + k-NN, warp per query) then K2b (plane fit + distance, thread per query)
// after_traversal (optional): recorded between K2a and K2b (nn_pos / nn_g2 are complete behind it)
// lm_pos / lm_m (optional, plane index only): K2a also answers BuildProblem's 1-NN of the map points of candidate 0 (LmState::nnb_pos /
// nbb_m), so that k_lm_knn_b need not run
cudaError_t launch_align3d(const DevPack &pk, const DevWork &wk, const DevParams &pr, int B, int debug, cudaStream_t st,
                           cudaEvent_t after_traversal = nullptr, uint32_t *lm_pos = nullptr, int *lm_m = nullptr);
cudaError_t launch_knn3d(const DevPack &pk, int kf, const double *d_q, int nq, int k, double radius2, uint32_t *d_idx, double *d_d2,
                         int *d_cnt, cudaStream_t st);

// the eigen-solver's correctly rounded acos / cos (crmath.cuh), element-wise: for the parity test against glibc
cudaError_t launch_debug_trig(const double *d_x, int n, double *d_acos, double *d_cos, cudaStream_t st);

// ---- K3 (reduce.cu) ----------------------------------------------------------------
// out: [B][out_stride] fp64 (first STL_EVAL_NSUMS of each row), written (not accumulated); out_stride 0 = STL_EVAL_NSUMS
// p2p (optional): the kernel also exchanges and sums each candidate's record over the ranks (p2p.cuh)
cudaError_t launch_reduce(const DevPack &pk, const DevWork &wk, const DevParams &pr, int B, double *d_out, cudaStream_t st, int out_stride = 0,
                          const P2pView *p2p = nullptr);
// stl_eval_frames: the per-keyframe records (stl_debug_frame's 13 values) of the selected keyframes of B candidates,
// d_out [B][n_kf][13] (rows of unselected keyframes untouched)
cudaError_t launch_frames(const DevPack &pk, const DevWork &wk, const DevParams &pr, int B, double *d_out, cudaStream_t st);

// ---- N4 (calib.cu): hand-eye initialisation edges and calibration-BA edges; HOST in, HOST out, synchronous
}  // namespace stl
struct stl_he_edges;
struct stl_calib_edges;
namespace stl {
cudaError_t he_linearize(const stl_he_edges &ed, const double *x, int B, double *h_out, double *h_chi2, cudaStream_t st);
cudaError_t calib_linearize(const stl_calib_edges &ed, const double *x, int B, double *h_out, double *h_chi2, cudaStream_t st);

}  // namespace stl
