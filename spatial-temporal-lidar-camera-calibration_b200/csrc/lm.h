// lm.h — LM path (Ceres / g2o side of the boundary): frozen residual blocks + linearisation.
#pragma once
#include "kernels.h"

namespace stl {

// Residual blocks frozen by stl_associate (BuildProblem, src/examples/iba_local.cpp:145-323), for a PROBLEM SET: P independent
// associations, problem p frozen at its own x0[p] (stl_associate_multi; stl_associate is the set of one).
// One slot per map-point-carrying correspondence of the association pass (slot = mp_off[kf] + qi); problem p owns the slots
// [p * slot_stride, p * slot_stride + n_slots) of every per-problem array below, so that a global slot index g = p * slot_stride
// + slot addresses them all.  Dense index lists select the slots that carry a 3-D/2-D block (IBA_PlaneFactor) and a 3-D/3-D
// block (Point2Point_Factor / Point2Plane_Factor).
struct LmState {
    bool ready = false;
    int P = 0;                    // problems in the frozen set
    int P_cap = 0;                // problems the per-problem arrays have room for
    long long n_slots = 0;
    long long slot_stride = 0;    // n_slots rounded up to 16
    int sub = 4;                  // CTAs per keyframe of the association kernels (= DevWork::sub)
    // ---- per problem ([P][slot_stride] unless stated)
    int *slot_kf = nullptr;
    uint32_t *slot_kp = nullptr;
    uint8_t *flags = nullptr;     // one allocation (room for P_cap): flag2d | type3d | flag3d | flagG, each [P][slot_stride], then d_counts [P][4]
    size_t flags_bytes = 0;
    uint8_t *flag2d = nullptr;    // 1 = plane block
    uint8_t *type3d = nullptr;    // 0 none, 1 point-to-point, 2 point-to-plane
    uint8_t *flag3d = nullptr;    // type3d != 0
    double *geo2d = nullptr;      // [.][6]  p0 (scan point, LiDAR frame), n0 (normal)
    double *geo3d = nullptr;      // [.][9]  map point (camera frame, unscaled), query point, normal
    // IBA_GPRFactor blocks (use_gpr): flag and neighbour list by slot
    uint8_t *flagG = nullptr;
    uint32_t *gpr_nb = nullptr;   // [.][32]
    int *gpr_m = nullptr;
    double *gpr_hyper = nullptr;  // [.][2] per-block (sigma, l) fitted at association time (null: the per-problem values)
    int *d_counts = nullptr;      // [P][4] device: plane blocks, 3-D blocks, point-to-point among them, GPR blocks
    // the 3-D/2-D and GPR lists of ALL problems, concatenated in problem order, each problem's run in slot order (global slot
    // indices): problem p's run starts at the sum of the counts of problems 0..p-1
    int *idx2d = nullptr, *idxG = nullptr;   // [P * slot_stride]
    int *idx3d = nullptr;         // [n_slots] 3-D/3-D list of problem 0, on demand (lm_compact3d, stl_eval_blocks)
    bool idx3d_valid = false;
    bool clear_lanes = false;     // re-association of part of the set: the lanes clear their problem's flags and counts first
    int *h_counts = nullptr;      // pinned [P][4], valid behind counts_done
    cudaEvent_t counts_done = nullptr;
    bool counts_valid = false;    // n_blocks below mirrors the device counts
    long long *n_blocks = nullptr;  // host [P][4]: plane (3-D/2-D), point-to-point, point-to-plane, GPR (3-D/2-D)
    bool use_gpr = false;
    long long max_blocks = 0;     // upper bound of any problem's block count (map-point-carrying keypoints)
    // ---- association scratch, one lane per problem associated by the same launch ([lanes][n_slots]): lives only during an
    // association, so it is sized by the lanes of one launch (<= the workspace chunk), not by P
    int lane_cap = 0;
    int2 *amap = nullptr;         // [lane_cap] device: (workspace candidate slot, problem) of association lane blockIdx.y
    int2 lane0 = {0, 0};          // = amap[0], passed with the kernel arguments (lane 0 needs no dependent load)
    int2 *h_amap = nullptr;       // pinned staging of amap
    cudaEvent_t amap_done = nullptr;
    uint8_t *stage = nullptr;     // 1 = plane at the scan point passed the gates, 3-D search pending
    double *plane_a = nullptr;    // [.][4] normal + regression error at the scan point
    uint32_t *nnb_pos = nullptr;  // 1-NN of the map point (0xffffffff = beyond max_3d_dist)
    uint32_t *nbb = nullptr;      // [.][32] neighbour list of that point
    float4 *nbbx = nullptr;       // [32][lane_cap * n_slots] coordinates of those neighbours, transposed
    long long nbbx_stride = 0;
    int *nbb_m = nullptr;         // (-2 = same point as the associated one)
    double *nbb_last = nullptr;
    int *d_sel = nullptr;         // [2] totals of the two selects (the per-problem counts are in d_counts)
    void *d_tmp = nullptr;        // cub scratch
    size_t tmp_bytes = 0;
    // ---- linearisation
    double *partial = nullptr;    // [B][grid][kLinVals]
    long long partial_cap = 0;
    void *d_cand = nullptr;       // [B] LmCand, then [B] int problem of each candidate
    void *h_cand = nullptr;       // pinned
    int cand_cap = 0;
    cudaEvent_t h2d_done = nullptr;  // guards the pinned staging buffer against reuse while a copy is in flight
};

void lm_free(LmState &lm);
// Sizes the set for P problems and `lanes` association lanes (all-or-nothing: a failure frees everything, P_cap = 0)
cudaError_t lm_reserve(const DevPack &pk, const DevParams &pr, LmState &lm, int P, int lanes, cudaStream_t st);
// Starts a new set of P problems (lm_reserve, all flags and counts cleared) or, partial, the re-association of some problems of
// the current set (each lane of the following lm_associate calls clears its problem first).
cudaError_t lm_begin(const DevPack &pk, const DevParams &pr, LmState &lm, int P, bool partial, int lanes, cudaStream_t st);
// Association lanes of the next lm_associate: lane j associates problem lanes[j].y from the K1 result (correspondences) at
// workspace candidate slot lanes[j].x
cudaError_t lm_set_lanes(LmState &lm, const int2 *lanes, int n, cudaStream_t st);
// BuildProblem of the n lanes set by lm_set_lanes, all in the same launches (grid (n_sel * sub, n): the selected keyframes).
// hints: the workspace holds, at each lane's candidate slot, the 1-NN position an evaluation at the SAME extrinsic found for each
// map point (DevWork::nn_pos) and, with cert, its lower bound of the squared distance to any other scan point (nn_g2): they
// seed, or settle, the 3-D search.
// part: 0 = everything; 1 = up to the plane at the associated scan point (needs K1's result only); 2 = the rest (needs the
// hints, i.e. K2a, when given) — the overlapped step enqueues the two parts around a wait for K2a.
// nn_folded: LmState::nnb_pos / nbb_m of lane 0 were written by K2a (launch_align3d with lm_pos / lm_m): k_lm_knn_b is not launched
cudaError_t lm_associate(const DevPack &pk, const DevWork &wk, const DevParams &pr, LmState &lm, int n, cudaStream_t st, bool hints,
                         bool cert, int part = 0, bool nn_folded = false);
// The dense 3-D/2-D list of every problem (one select over the [P][slot_stride] flags): after part 1 of every lane
cudaError_t lm_compact2d(LmState &lm, cudaStream_t st);
// The dense GPR list (use_gpr) after the last lane; marks the set ready
cudaError_t lm_finish_associate(LmState &lm, bool use_gpr, cudaStream_t st);
// Block-count read-back behind lm.counts_done
cudaError_t lm_copy_counts(LmState &lm, cudaStream_t st);
// problem (optional, host [B]): the problem candidate b is linearised on (null: problem 0)
cudaError_t lm_stage_candidates(LmState &lm, const double *x, const int *problem, int B, cudaStream_t st);
// x: HOST [B][7]; d_out: DEVICE [B][STL_LIN_NSUMS]
// optional per-block output of a linearisation (device pointers; B must be 1)
struct BlockOut {
    int32_t *type = nullptr, *kf = nullptr, *kp = nullptr, *nres = nullptr;  // [n_blocks]
    double *res = nullptr;  // [n_blocks][rmax]
    double *jac = nullptr;  // [n_blocks][rmax][7]
    int rmax = 0;
};

// out_stride: doubles between the records of consecutive candidates in d_out (0 = STL_LIN_NSUMS)
// problem (optional, host [B]): as lm_stage_candidates; null: every candidate on problem 0, which the kernels then read from no index
cudaError_t lm_linearize(const DevPack &pk, const DevParams &pr, LmState &lm, const double *x, const int *problem, int B, double *d_out,
                         cudaStream_t st, const BlockOut *blocks = nullptr, int out_stride = 0, const P2pView *p2p = nullptr,
                         cudaEvent_t before_finish = nullptr, bool cand_staged = false);
cudaError_t lm_compact3d(const DevPack &pk, LmState &lm, cudaStream_t st);
// cand_staged: the caller has already run lm_stage_candidates(lm, x, problem, B, st) for exactly these x on this stream
// before_finish (optional): event the finishing kernel waits for (the rest of the record it completes / exchanges)
// waits for the last association and mirrors its block counts into lm.n_blocks
cudaError_t lm_block_counts(LmState &lm);
// GPR::fit for every GPR block of problem p (IBA_GPRFactor's constructor, IBACalib2.hpp:441-461): the training pixels / depths
// are formed on the device with the association extrinsic c0 (device), the two-parameter fit runs on the host (OpenMP over
// blocks), the result lands in lm.gpr_hyper.  Synchronous.
cudaError_t lm_fit_gpr_hyper(const DevPack &pk, const DevCand *c0, const DevParams &pr, LmState &lm, int p, cudaStream_t st, int flavour);
// copies (sigma, l) of the GPR blocks of problem 0, block order, to host memory out[nG][2]
cudaError_t lm_get_gpr_hyper(const DevParams &pr, LmState &lm, double *out, cudaStream_t st);

}  // namespace stl
