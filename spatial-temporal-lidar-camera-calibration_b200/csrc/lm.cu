// lm.cu — the Levenberg-Marquardt side of the boundary.
//
// K4a  k_lm_associate: BuildProblem (src/examples/iba_local.cpp:145-323) — for every 2-D
//      correspondence of the association pass (K1 at the current estimate):
//        ComputeLocalNeighbor            include/pointcloud.h:733-760   (iba_local.cpp:207)
//        plane fit + regression gate     iba_local.cpp:218-231
//        covisible observations          iba_local.cpp:245-259
//        map point -> LiDAR, 1-NN gate   iba_local.cpp:239-240,283-290
//        ComputeLocalNormalSingleThre    include/pointcloud.h:699-717,651-666 (iba_local.cpp:295)
//      and freezes the residual blocks on the device.
// K4b  k_linearize: evaluates the frozen blocks at B parameter vectors —
//        IBA_PlaneFactor::operator()     include/IBACalib2.hpp:152-184 (g2o twin IBACalib.hpp:103-140)
//        Point2Point_Factor              include/IBACalib2.hpp:570-584
//        Point2Plane_Factor              include/IBACalib2.hpp:611-625
//      with the Jet evaluation's values and chain-rule partials (linrow.cuh), ceres::HuberLoss + Corrector semantics
//      (iba_local.cpp:263,291; rho'' <= 0 => residual and Jacobian scaled by sqrt(rho')),
//      and reduces cost, J^T r and the 7x7 J^T J in fp64 (warp shuffles, fixed order).
#include <cub/cub.cuh>

#include "../../include/stlcalib.h"
#include "dual.cuh"
#include "gprfit.hpp"
#include "knn.cuh"
#include "linrow.cuh"
#include "lm.h"

namespace stl {
namespace {

constexpr int kWarps = 8;
#ifndef STL_LM_MINB
#define STL_LM_MINB 6  // resident CTAs per SM of the association's traversal kernels (40 registers): 8 / 6 / 5 measured 0.216 / 0.198 / 0.195 ms for the stage
#endif
// CTAs per keyframe of the association kernels: LmState::sub, chosen from the keyframe count of the pack (4 at the KITTI-00
// shape; more for a small keyframe shard of a multi-GPU run, whose few keyframes would otherwise leave most SMs idle)
constexpr int kLinVals = 41;  // cost, g[7], H upper 28, n2d, npt, npl, nres, ngpr
constexpr int kGprWarps = 1;  // one warp per CTA: the dual kernel matrix of a block takes ~40 KB of shared memory
constexpr int kLinThreads = 128;

// ------------------------------------------------------------------ K4a (four small kernels)
// All four walk the correspondences that carry a map point (the query list K1 wrote), keyframe by
// keyframe; list slot = block slot = mp_off[f] + qi.  Traversals are warp-per-item, plane fits thread-per-item.
// With the plane index only k_lm_plane_a and k_lm_plane_b run (and inside stl_step_batch K2a answers k_lm_knn_b's question).
// grid (n_sel * sub, lanes) over the keyframe selection (DevPack::sel; all keyframes without one): association lane blockIdx.y reads the K1 result at its workspace candidate slot, works in its own
// scratch and writes the arrays of its problem (lm_lane) — a lane computes exactly what a single association computes.

// Narrows the workspace, the scratch and the problem arrays to association lane blockIdx.y.
// arg0: lane 0 takes its map from the kernel arguments (lm.lane0 == amap[0], lm_set_lanes) instead of a dependent load
// (k_lm_plane_b reads amap: the argument copy costs it a register spill)
__device__ __forceinline__ void lm_lane(const DevPack &pk, DevWork &wk, LmState &lm, bool arg0 = true) {
    const int2 am = arg0 && blockIdx.y == 0 ? lm.lane0 : lm.amap[blockIdx.y];
    const long long nk = pk.n_kp_total, F = pk.n_kf, nm = lm.n_slots;
    const long long wc = am.x, wq = wc * nm;
    wk.cand += wc;
    wk.corr_kp += wc * nk; wk.corr_sp += wc * nk; wk.q_corr += wc * nk; wk.q_kpsp += wc * nk;
    wk.n_corr += wc * F; wk.n_q += wc * F;
    wk.nn_pos += wq; wk.nn_g2 += wq; wk.nb += wq * kMaxK; wk.nbx += wq; wk.nb_m += wq; wk.nb_last += wq;
    const long long lo = (long long)blockIdx.y * nm;
    lm.stage += lo; lm.plane_a += lo * 4; lm.nnb_pos += lo; lm.nbb += lo * kMaxK; lm.nbbx += lo; lm.nbb_m += lo; lm.nbb_last += lo;
    const long long po = (long long)am.y * lm.slot_stride;
    lm.slot_kf += po; lm.slot_kp += po; lm.flag2d += po; lm.type3d += po; lm.flag3d += po; lm.flagG += po;
    lm.geo2d += po * 6; lm.geo3d += po * 9; lm.gpr_nb += po * kMaxK; lm.gpr_m += po;
    lm.d_counts += am.y * 4;
}

// clears the flags and counts of the problem of every lane (re-association of part of a set)
__global__ void k_lm_clear(LmState lm) {
    const long long po = (long long)lm.amap[blockIdx.y].y * lm.slot_stride, n = lm.slot_stride, ptot = (long long)lm.P * n;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        lm.flags[po + i] = 0; lm.flags[ptot + po + i] = 0; lm.flags[2 * ptot + po + i] = 0; lm.flags[3 * ptot + po + i] = 0;
    }
    if (blockIdx.x == 0 && threadIdx.x < 4) lm.d_counts[lm.amap[blockIdx.y].y * 4 + threadIdx.x] = 0;
}

__device__ __forceinline__ bool lm_frame_active(const DevWork &wk, const DevParams &pr, int f, int &nq) {
    nq = wk.n_q[f];
    return wk.n_corr[f] >= pr.num_min_corr && nq > 0;  // iba_local.cpp:192
}

// map point in the reference camera frame, no scale (iba_local.cpp:239-240)
__device__ __forceinline__ void lm_map_point(const DevPack &pk, const DevKf &K, int f, uint32_t kp, double &Mx, double &My, double &Mz) {
    const float *Tcw = pk.Tcw + (long long)f * 12;
    const float *mp = pk.kp_mp + (K.kp_off + kp) * 3;
    const double a = (double)mp[0], b = (double)mp[1], c = (double)mp[2];
    Mx = dadd(dot3e((double)Tcw[0], (double)Tcw[1], (double)Tcw[2], a, b, c), (double)Tcw[3]);
    My = dadd(dot3e((double)Tcw[4], (double)Tcw[5], (double)Tcw[6], a, b, c), (double)Tcw[7]);
    Mz = dadd(dot3e((double)Tcw[8], (double)Tcw[9], (double)Tcw[10], a, b, c), (double)Tcw[11]);
}

// L1: ComputeLocalNeighbor around the associated scan point (pointcloud.h:733-760, iba_local.cpp:207).
// The reference searches for every correspondence and only afterwards drops those without a map
// point (:213) or without a covisible observation (:259); neither test depends on the search, so
// they come first here.
__global__ void __launch_bounds__(kWarps * 32, STL_LM_MINB)
k_lm_knn_a(const DevPack pk, DevWork wk, const DevParams pr, LmState lm) {
    lm_lane(pk, wk, lm);
    const int j = blockIdx.x % lm.sub, f = sel_kf(pk, blockIdx.x / lm.sub);
    int nq;
    if (!lm_frame_active(wk, pr, f, nq)) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const DevKf K = pk.kf[f];
    const ScanView S = make_view(pk, K);
    const int C = pk.n_covis;
    __shared__ int ticket;
    if (threadIdx.x == 0) ticket = 0;
    __syncthreads();
    for (;;) {
        const int qi = next_ticket(&ticket, lane) * lm.sub + j;
        if (qi >= nq) break;
        const uint2 ks = wk.q_kpsp[K.kp_off + qi];
        const uint32_t kp = ks.x, sp = ks.y;
        const long long slot = K.mp_off + qi;
        // lane s looks at covisible keyframe s (C <= STL_MAX_COVIS <= 32)
        const bool obs = lane < C && pk.covis_valid[f * C + lane] && !isnan(pk.covis_uv[(K.kp_off + kp) * C + lane].x);
        const int ncov = __popc(__ballot_sync(kFull, obs));
        if (ncov == 0) {  // iba_local.cpp:259
            if (lane == 0) wk.nb_m[slot] = -1;
            continue;
        }
        if (pr.plane_index && !pr.use_gpr) {  // the plane of the scan point comes from the index
            if (lane == 0) wk.nb_m[slot] = 0;
            continue;
        }
        SinkK kn(pr.k, pr.radius2);
        knn_around_point(S, sp, kn, lane);
        wk.nb[slot * kMaxK + lane] = lane < kn.count ? kn.kpos : 0xffffffffu;
        store_nb_coords(wk.nbx, wk.nbx_stride, slot, S, lane, kn.count, kn.kpos);
        const double last = __shfl_sync(kFull, kn.kd, kn.count > 0 ? kn.count - 1 : 0);
        if (lane == 0) { wk.nb_m[slot] = kn.count; wk.nb_last[slot] = last; }
    }
}

// L2: plane at the scan point (iba_local.cpp:218-231) -> 3-D/2-D block; decides whether the 3-D search runs
__global__ void __launch_bounds__(128)
k_lm_plane_a(const DevPack pk, DevWork wk, const DevParams pr, LmState lm) {
    lm_lane(pk, wk, lm);
    const int j = blockIdx.x % lm.sub, f = sel_kf(pk, blockIdx.x / lm.sub);
    int nq;
    if (!lm_frame_active(wk, pr, f, nq)) return;
    __shared__ int cnt[2];  // plane blocks, GPR blocks of this CTA (one pair of global atomics per CTA)
    if (threadIdx.x < 2) cnt[threadIdx.x] = 0;
    __syncthreads();
    const DevKf K = pk.kf[f];
    const ScanView S = make_view(pk, K);
    const bool from_index = pr.plane_index && !pr.use_gpr;  // then k_lm_knn_a did not run: the covisibility test is made here
    const int C = pk.n_covis;
    for (int qi = j * blockDim.x + threadIdx.x; qi < nq; qi += lm.sub * blockDim.x) {
        const long long slot = K.mp_off + qi;
        lm.stage[slot] = 0;
        const uint32_t ci = wk.q_corr[K.kp_off + qi];
        const uint32_t kp = wk.corr_kp[K.kp_off + ci], sp = wk.corr_sp[K.kp_off + ci];
        int m = 0;
        if (from_index) {
            bool any = false;
            for (int s = 0; s < C; ++s) any = any || (pk.covis_valid[f * C + s] && !isnan(pk.covis_uv[(K.kp_off + kp) * C + s].x));
            if (!any) continue;  // iba_local.cpp:259
        } else {
            m = wk.nb_m[slot];
            if (m < 0) continue;
        }
        const double cx = (double)S.px[sp], cy = (double)S.py[sp], cz = (double)S.pz[sp];
        const PlaneOut po = from_index ? plane_lookup(pk, K, sp)
                                       : plane_fit(NbCoords{wk.nbx + slot, wk.nbx_stride}, m, wk.nb_last[slot], cx, cy, cz, pr);
        if (!po.gates_ok) continue;  // m < min_pts || d2[m-1] < min_diff^2 (pointcloud.h:754)
        const long long cs = slot;  // block slot = query slot (the only keypoints that can carry a block are those with a map point)
        lm.slot_kf[cs] = f;
        lm.slot_kp[cs] = kp;
        double *pa = lm.plane_a + slot * 4;
        pa[0] = po.n.x; pa[1] = po.n.y; pa[2] = po.n.z; pa[3] = po.reg;
        if (po.reg < pr.reg_thr) {  // strict '<' (iba_local.cpp:231)
            double *g = lm.geo2d + cs * 6;
            g[0] = cx; g[1] = cy; g[2] = cz; g[3] = po.n.x; g[4] = po.n.y; g[5] = po.n.z;
            lm.flag2d[cs] = 1;
            atomicAdd(&cnt[0], 1);
        } else if (pr.use_gpr) {
            // non-planar neighbourhood: IBA_GPRFactor over the neighbour points (iba_local.cpp:272-280);
            // the list is copied because the evaluation workspace is reused by later calls
            for (int t = 0; t < kMaxK; ++t) lm.gpr_nb[slot * kMaxK + t] = wk.nb[slot * kMaxK + t];
            lm.gpr_m[slot] = po.m;
            lm.flagG[cs] = 1;
            atomicAdd(&cnt[1], 1);
        }
        lm.stage[slot] = 1;
    }
    __syncthreads();
    if (threadIdx.x < 2 && cnt[threadIdx.x] > 0) atomicAdd(lm.d_counts + 3 * threadIdx.x, cnt[threadIdx.x]);  // [0] plane, [3] GPR
}

// L3: map point -> LiDAR frame with the association extrinsic, 1-NN gate, neighbourhood of that point
// (iba_local.cpp:283-295).
// A warp draws 32 queries at a time, one per lane.  When the evaluation at this same extrinsic has just answered the 1-NN
// of the map point's float32-scaled twin q (K2a: position h, and g2 = a lower bound of the squared distance from q to every
// OTHER scan point), the LM query q' — the same map point scaled in fp64, a few micrometres from q — needs no search if
//     sqrt(g2) - |q - q'|  >  |q' - h|                                  (triangle inequality, margins below):
// every other point is then strictly farther from q' than h, so h is exactly what the KD-tree search returns.  Lanes
// whose query is not settled that way (no evaluation at hand, near-equidistant neighbours) take turns on the warp-wide
// exact search, seeded with h or with the associated scan point.
__global__ void __launch_bounds__(kWarps * 32, STL_LM_MINB)
k_lm_knn_b(const DevPack pk, DevWork wk, const DevParams pr, LmState lm, const bool hints, const bool cert) {
    lm_lane(pk, wk, lm);
    const uint32_t *__restrict__ nn_hint = hints ? wk.nn_pos : nullptr;
    const float *__restrict__ nn_g2 = hints && cert ? wk.nn_g2 : nullptr;
    const int j = blockIdx.x % lm.sub, f = sel_kf(pk, blockIdx.x / lm.sub);
    int nq;
    if (!lm_frame_active(wk, pr, f, nq)) return;
    const int lane = threadIdx.x & 31;
    const DevKf K = pk.kf[f];
    const DevCand &c0 = wk.cand[0];
    const ScanView S = make_view(pk, K);
    const float *Tcw = pk.Tcw + (long long)f * 12;
    __shared__ int ticket;
    if (threadIdx.x == 0) ticket = 0;
    __syncthreads();
    for (;;) {
        const int base = next_ticket(&ticket, lane) * 32;
        if ((long long)base * lm.sub + j >= nq) break;
        const int qi = (base + lane) * lm.sub + j;
        const long long slot = K.mp_off + qi;
        const bool valid = qi < nq && lm.stage[slot] == 1;
        uint32_t sp = 0, hint = 0xffffffffu, nn_pos = 0xffffffffu;
        double qx = 0, qy = 0, qz = 0, nn_d = DBL_MAX;
        bool settled = false;
        if (valid) {
            const uint2 ks = wk.q_kpsp[K.kp_off + qi];
            const uint32_t kp = ks.x;
            sp = ks.y;
            double Mx, My, Mz;
            lm_map_point(pk, K, f, kp, Mx, My, Mz);
            xform(c0.Ri, c0.ti, dmul(Mx, c0.s), dmul(My, c0.s), dmul(Mz, c0.s), qx, qy, qz);  // initSE3.inverse() * (MapPoint * init_scale)
            hint = nn_hint ? nn_hint[slot] : sp;
            if (hint == 0xffffffffu) hint = sp;
            if (nn_hint && nn_g2 && nn_hint[slot] != 0xffffffffu) {
                // the evaluation's query for this map point (iba_global.cpp:231-234: GetWorldPos() * scale in float32)
                const float *mp = pk.kp_mp + (K.kp_off + kp) * 3;
                const double wx = (double)__fmul_rn(mp[0], c0.sf), wy = (double)__fmul_rn(mp[1], c0.sf), wz = (double)__fmul_rn(mp[2], c0.sf);
                const double ex = dadd(dot3e((double)Tcw[0], (double)Tcw[1], (double)Tcw[2], wx, wy, wz), dmul((double)Tcw[3], c0.s));
                const double ey = dadd(dot3e((double)Tcw[4], (double)Tcw[5], (double)Tcw[6], wx, wy, wz), dmul((double)Tcw[7], c0.s));
                const double ez = dadd(dot3e((double)Tcw[8], (double)Tcw[9], (double)Tcw[10], wx, wy, wz), dmul((double)Tcw[11], c0.s));
                double ox, oy, oz;
                xform(c0.Ri, c0.ti, ex, ey, ez, ox, oy, oz);
                const double move = sqrt(dist3e(ox, oy, oz, qx, qy, qz)) * (1.0 + 1e-9) + 1e-12;  // |q - q'|, rounded up
                const double dh = dist3e(qx, qy, qz, (double)S.px[hint], (double)S.py[hint], (double)S.pz[hint]);
                const double reach = (double)__fsqrt_rd(nn_g2[slot]) - move;                      // every other point is at least this far from q'
                if (reach > 0.0 && reach * reach > dh * (1.0 + 1e-6) + 1e-18) { settled = true; nn_pos = hint; nn_d = dh; }
            }
        }
        // exact searches for the lanes that are not settled, one query at a time on the whole warp
        unsigned todo = __ballot_sync(kFull, valid && !settled);
        while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            const double sx = __shfl_sync(kFull, qx, src), sy = __shfl_sync(kFull, qy, src), sz = __shfl_sync(kFull, qz, src);
            const uint32_t sh = __shfl_sync(kFull, hint, src);
            Sink1 nn;
            nn_near_leaf(S, pr.adj_r, (int)(sh >> 5), sx, sy, sz, nn, lane, sh);
            if (lane == src) { nn_pos = nn.pos; nn_d = nn.d; }
        }
        bool want_knn = false;
        if (valid) {
            if (nn_d > pr.max_3d_dist2) {  // iba_local.cpp:289
                lm.nnb_pos[slot] = 0xffffffffu;
            } else {
                lm.nnb_pos[slot] = nn_pos;
                if (nn_pos == sp) lm.nbb_m[slot] = -2;          // very often the associated scan point itself: its plane is already known
                else if (pr.plane_index) lm.nbb_m[slot] = -3;   // looked up by k_lm_plane_b
                else want_knn = true;
            }
        }
        unsigned kn_todo = __ballot_sync(kFull, want_knn);
        while (kn_todo) {
            const int src = __ffs(kn_todo) - 1;
            kn_todo &= kn_todo - 1;
            const uint32_t p = __shfl_sync(kFull, nn_pos, src);
            const long long sl = K.mp_off + ((long long)(base + src) * lm.sub + j);
            SinkK kn(pr.k, pr.radius2);
            knn_around_point(S, p, kn, lane);
            lm.nbb[sl * kMaxK + lane] = lane < kn.count ? kn.kpos : 0xffffffffu;
            store_nb_coords(lm.nbbx, lm.nbbx_stride, sl, S, lane, kn.count, kn.kpos);
            const double last = __shfl_sync(kFull, kn.kd, kn.count > 0 ? kn.count - 1 : 0);
            if (lane == 0) { lm.nbb_m[sl] = kn.count; lm.nbb_last[sl] = last; }
        }
    }
}

// L4: ComputeLocalNormalSingleThre at the map point's neighbour (pointcloud.h:699-717,651-666) -> 3-D/3-D block.
// Geometry of the 3-D/3-D block of query slot `slot` (keyframe f, keypoint kp): g = map point (camera frame, unscaled), its
// nearest scan point, the plane normal there; type 1 = Point2Point_Factor, 2 = Point2Plane_Factor (iba_local.cpp:300-309).
// False: the slot carries no such block.
__device__ __forceinline__ bool block3d_geometry(const DevPack &pk, const DevParams &pr, const LmState &lm, long long slot, int f, uint32_t kp,
                                                 double g[9], int &type) {
    if (lm.stage[slot] != 1) return false;
    const uint32_t np = lm.nnb_pos[slot];
    if (np == 0xffffffffu) return false;
    const DevKf &K = pk.kf[f];
    const float *sx = pk.px + K.pt_off, *sy = pk.py + K.pt_off, *sz = pk.pz + K.pt_off;
    const double nx = (double)sx[np], ny = (double)sy[np], nz = (double)sz[np];
    bool gates_ok, state;
    double n3[3];
    const int m = lm.nbb_m[slot];
    if (m == -2) {
        const double *pa = lm.plane_a + slot * 4;
        gates_ok = true; n3[0] = pa[0]; n3[1] = pa[1]; n3[2] = pa[2];
        state = pa[3] < pr.reg_thr;
    } else {
        const PlaneOut p2 = m == -3 ? plane_lookup(pk, K, np) : plane_fit(NbCoords{lm.nbbx + slot, lm.nbbx_stride}, m, lm.nbb_last[slot], nx, ny, nz, pr);
        gates_ok = p2.gates_ok; n3[0] = p2.n.x; n3[1] = p2.n.y; n3[2] = p2.n.z;
        state = p2.gates_ok && p2.reg < pr.reg_thr;
    }
    lm_map_point(pk, K, f, kp, g[0], g[1], g[2]);
    g[3] = nx; g[4] = ny; g[5] = nz;
    g[6] = gates_ok ? n3[0] : 0.0; g[7] = gates_ok ? n3[1] : 0.0; g[8] = gates_ok ? n3[2] : 1.0;
    type = state ? 2 : 1;
    return true;
}

__global__ void __launch_bounds__(128)
k_lm_plane_b(const DevPack pk, DevWork wk, const DevParams pr, LmState lm) {
    lm_lane(pk, wk, lm, false);
    const int j = blockIdx.x % lm.sub, f = sel_kf(pk, blockIdx.x / lm.sub);
    int nq;
    if (!lm_frame_active(wk, pr, f, nq)) return;
    const DevKf K = pk.kf[f];
    __shared__ int cnt[2];  // blocks of this CTA: all, point-to-point (one pair of global atomics per CTA, not per block)
    if (threadIdx.x < 2) cnt[threadIdx.x] = 0;
    __syncthreads();
    for (int qi = j * blockDim.x + threadIdx.x; qi < nq; qi += lm.sub * blockDim.x) {
        const long long slot = K.mp_off + qi;
        if (lm.stage[slot] != 1) continue;
        if (lm.nnb_pos[slot] == 0xffffffffu) continue;
        const uint32_t ci = wk.q_corr[K.kp_off + qi];
        const uint32_t kp = wk.corr_kp[K.kp_off + ci];
        double g9[9];
        int type;
        if (!block3d_geometry(pk, pr, lm, slot, f, kp, g9, type)) continue;
        double *g = lm.geo3d + slot * 9;
#pragma unroll
        for (int i = 0; i < 9; ++i) g[i] = g9[i];
        lm.type3d[slot] = (uint8_t)type;
        lm.flag3d[slot] = 1;
        atomicAdd(&cnt[0], 1);                    // 3-D/3-D blocks  (integer counts: the order does not matter)
        if (type == 1) atomicAdd(&cnt[1], 1);     // point-to-point blocks among them
    }
    __syncthreads();
    if (threadIdx.x < 2 && cnt[threadIdx.x] > 0) atomicAdd(lm.d_counts + 1 + threadIdx.x, cnt[threadIdx.x]);
}

// ------------------------------------------------------------------ K4b
struct Acc {
    double v[kLinVals];
};

__device__ __forceinline__ void huber(double sq, double delta, double &rho0, double &sr) {
    if (sq > delta * delta) {  // ceres::HuberLoss::Evaluate
        const double r = sqrt(sq);
        rho0 = 2.0 * delta * r - delta * delta;
        sr = sqrt(fmax(DBL_MIN, delta / r));
    } else {
        rho0 = sq;
        sr = 1.0;
    }
}

__device__ __forceinline__ void accumulate(Acc &A, const D7 &e, double sr) {
    const double r = sr * e.a;
    double J[7];
#pragma unroll
    for (int a = 0; a < 7; ++a) J[a] = sr * e.v[a];
    int h = 8;
#pragma unroll
    for (int a = 0; a < 7; ++a) {
        A.v[1 + a] += J[a] * r;
#pragma unroll
        for (int b = a; b < 7; ++b) A.v[h++] += J[a] * J[b];
    }
}

__device__ __forceinline__ void mv3(const D7 *M, const D7 *p, D7 *o) {
#pragma unroll
    for (int i = 0; i < 3; ++i) o[i] = (M[i * 3] * p[0] + M[i * 3 + 1] * p[1]) + M[i * 3 + 2] * p[2];
}
// k_linearize's rows (linrow.cuh): J^T r and J^T J by fused multiply-adds
__device__ __forceinline__ void accumulate(Acc &A, const Row7 &e, double sr) {
    const double r = sr * e.a;
    double J[7];
#pragma unroll
    for (int a = 0; a < 7; ++a) J[a] = sr * e.v[a];
    int h = 8;
#pragma unroll
    for (int a = 0; a < 7; ++a) {
        A.v[1 + a] = fma(J[a], r, A.v[1 + a]);
#pragma unroll
        for (int b = a; b < 7; ++b) { A.v[h] = fma(J[a], J[b], A.v[h]); ++h; }
    }
}

// Optional per-block output (stl_eval_blocks): what a Ceres CostFunction::Evaluate / a g2o edge would
// return for each frozen residual block — raw residuals and their 7-column Jacobian rows, no robust
// kernel (the solver applies its own loss).  Fixed stride of rmax rows per block.
template <class T7>
__device__ __forceinline__ void put_row(const BlockOut &o, long long blk, int r, const T7 &e) {
    o.res[blk * o.rmax + r] = e.a;
    double *j = o.jac + (blk * o.rmax + r) * 7;
#pragma unroll
    for (int a = 0; a < 7; ++a) j[a] = e.v[a];
}
__device__ __forceinline__ void put_head(const BlockOut &o, long long blk, int type, int kf, uint32_t kp, int nres) {
    o.type[blk] = type; o.kf[blk] = kf; o.kp[blk] = (int32_t)kp; o.nres[blk] = nres;
}

// Start of problem p's run in a concatenated block list: the sum of the counts `which` of problems 0..p-1 (warp 0 of the CTA;
// integer sums, so the order does not matter)
__device__ __forceinline__ void lm_list_start(const LmState &lm, int p, int which, int *out) {
    if (threadIdx.x >= 32) return;
    int s = 0;
    for (int q = threadIdx.x; q < p; q += 32) s += lm.d_counts[q * 4 + which];
    for (int o = 16; o; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    if (threadIdx.x == 0) *out = s;
}

// x, re-read: the address carries an offset of zero the compiler cannot see through, so loads from x inside a loop are not
// hoisted out of it.  k_linearize reads its candidate tables (~190 doubles, shared memory) through this once per block: kept in
// registers across the block loops they spill.
template <class T>
__device__ __forceinline__ const T &reread(const T &x) {
    int z;
    asm volatile("mov.b32 %0, 0;" : "=r"(z));
    return *reinterpret_cast<const T *>(reinterpret_cast<const char *>(&x) + z);
}

// Problem-local slot of slot v of the selection's compacted slot range (DevPack::sel_mp): with a keyframe selection the 3-D walk
// runs over the selected keyframes' slots only, grouped 32 at a time as a pack of those keyframes groups them, so that every
// thread sums the blocks it would sum there
__device__ __forceinline__ int sel_slot(const DevPack &pk, int v) {
    int lo = 0, hi = pk.n_sel;  // sel_mp[lo].x <= v < sel_mp[hi].x
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (pk.sel_mp[mid].x <= v) lo = mid; else hi = mid;
    }
    return v + pk.sel_mp[lo].y;
}


// First position in the sorted run l[0, n) whose value is >= v
__device__ __forceinline__ int lower_pos(const int *__restrict__ l, int n, long long v) {
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (l[mid] < v) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// grid (chunks, B): candidate blockIdx.y on problem cprob[blockIdx.y].  The 3-D/3-D blocks are walked over ALL query slots of
// that problem (no compacted list: the work per block is light, and the association then has no select on the way to the
// linearisation).  WB (stl_eval_blocks) numbers the blocks and therefore walks the compacted list (problem 0).
// MINB: resident CTAs per SM the registers must allow (lm_linearize); the two forms compute the same bits.
// FR (stl_linearize_frames): per-keyframe rows, grid (ceil(n_sel / 4), B).  Warp w of CTA x sums the blocks of selection position
// x * 4 + w alone, the four warps sharing the candidate tables: its 3-D/2-D blocks are the keyframe's run of the problem's idx2d
// list (slot order, found by binary search for the keyframe's slot bounds), lane l taking the run's blocks l, l + 32, ...; its
// 3-D/3-D blocks come from the queue walk below over the keyframe's own slots [mp_off, mp_off + n_mp), 32 per round; the warp's
// shuffle tree makes the row, written at partial[blockIdx.y][position] (partial_stride = n_sel).  Which lane sums which block,
// and the order of the sum, so depend on the keyframe's blocks alone: not on B, the other candidates, the selection, the problem
// set or the shard holding the keyframe.
template <bool WB, int MINB, bool FR = false>
__global__ void __launch_bounds__(kLinThreads, MINB)
k_linearize(const DevPack pk, const DevParams pr, const LmState lm, const LmCand *__restrict__ cands, const int *__restrict__ cprob,
            double *__restrict__ partial, int partial_stride, const BlockOut bo) {
    __shared__ LmCand c;
    __shared__ double W[9][7];  // candidate table of the 3-D/3-D partials (linrow.cuh)
    __shared__ int list0;
    const int prob = cprob ? cprob[blockIdx.y] : 0;
    {
        const double *src = reinterpret_cast<const double *>(cands + blockIdx.y);
        double *dst = reinterpret_cast<double *>(&c);
        for (int i = threadIdx.x; i < (int)(sizeof(LmCand) / 8); i += kLinThreads) dst[i] = src[i];
        lin_table(cands[blockIdx.y], W, threadIdx.x, kLinThreads);
    }
    lm_list_start(lm, prob, 0, &list0);
    __syncthreads();
    const int fpos = FR ? (int)(blockIdx.x * (kLinThreads / 32) + (threadIdx.x >> 5)) : 0;  // FR: the warp's selection position
    if (FR && fpos >= pk.n_sel) return;  // whole warps; FR has no CTA barrier below
    Acc A;
#pragma unroll
    for (int i = 0; i < kLinVals; ++i) A.v[i] = 0.0;
    const int C = pk.n_covis;
    const int stride = FR ? 32 : gridDim.x * kLinThreads;
    long long s0 = 0, s1 = 0;  // FR: the keyframe's problem-local slots
    if (FR) {
        const DevKf &Kf = pk.kf[sel_kf(pk, fpos)];
        s0 = Kf.mp_off;
        s1 = Kf.mp_off + Kf.n_mp;
    }

    // block counts live on the device (written by the association kernels on this stream): no host round trip
    const int *counts = lm.d_counts + prob * 4;
    const int n2d_all = counts[0];
    const int *idx2d = lm.idx2d + list0;
    const long long pg = (long long)prob * lm.slot_stride;
    const int t0 = FR ? lower_pos(idx2d, n2d_all, pg + s0) + (int)(threadIdx.x & 31) : blockIdx.x * kLinThreads + threadIdx.x;
    const int n2d = FR ? lower_pos(idx2d, n2d_all, pg + s1) : n2d_all;
    // ---- 3-D/2-D blocks: IBA_PlaneFactor (IBACalib2.hpp:152-184)
    for (int it = t0; it < n2d; it += stride) {
        const int slot = idx2d[it];  // global slot (problem offset included)
        const LmCand &cb = reread(c);
        const int f = lm.slot_kf[slot];
        const uint32_t kp = lm.slot_kp[slot];
        const DevKf &K = pk.kf[f];
        const double fx = K.fx, fy = K.fy, cx = K.cx, cy = K.cy;
        const float2 kxy = pk.kp_xy[K.kp_off + kp];
        double g[6];
#pragma unroll
        for (int i = 0; i < 6; ++i) g[i] = lm.geo2d[(long long)slot * 6 + i];
        const double Cxz = ((double)kxy.x - cx) / fx, Cyz = ((double)kxy.y - cy) / fy;
        double Z0, dZ[7];
        p2_depth(cb, g, Cxz, Cyz, Z0, dZ);
        // pass 1: squared norm of the block (values only) for the robust kernel
        double sq = 0.0;
        int nres = 0;
        for (int s = 0; s < C; ++s) {
            if (!pk.covis_valid[f * C + s]) continue;
            const float2 uv = pk.covis_uv[(K.kp_off + kp) * C + s];
            if (isnan(uv.x)) continue;
            const float *rp = pk.relpose + ((long long)f * C + s) * 12;
            double P1[3];
            p2_point(cb, rp, Z0, Cxz, Cyz, P1);
            const double eu = (fx * P1[0] / P1[2] + cx) - (double)uv.x, ev = (fy * P1[1] / P1[2] + cy) - (double)uv.y;
            sq += eu * eu;
            sq += ev * ev;
            nres += 2;
        }
        double rho0, sr;
        huber(sq, pr.delta2d, rho0, sr);
        A.v[0] += 0.5 * rho0;
        A.v[36] += 1.0;
        A.v[39] += (double)nres;
        // pass 2: the rows with their partials
        int wrow = 0;
        for (int s = 0; s < C; ++s) {
            if (!pk.covis_valid[f * C + s]) continue;
            const float2 uv = pk.covis_uv[(K.kp_off + kp) * C + s];
            if (isnan(uv.x)) continue;
            const float *rp = pk.relpose + ((long long)f * C + s) * 12;
            double P1[3];
            p2_point(cb, rp, Z0, Cxz, Cyz, P1);
            Row7 eu, ev;
            p2_rows(cb, rp, P1, dZ, Cxz, Cyz, fx, fy, cx, cy, uv.x, uv.y, eu, ev);
            accumulate(A, eu, sr);
            accumulate(A, ev, sr);
            if (WB) { put_row(bo, it, wrow, eu); put_row(bo, it, wrow + 1, ev); wrow += 2; }
        }
        if (WB) put_head(bo, it, 0, f, kp, nres);
    }

    // ---- 3-D/3-D blocks: Point2Point_Factor / Point2Plane_Factor (IBACalib2.hpp:570-584,611-625)
    // WB: the compacted list (numbered blocks), one block per thread and round.  Otherwise every warp walks 32 consecutive query
    // slots per round, queues the flagged ones in shared memory and evaluates 32 queued blocks at a time (the tail at the end): the
    // lanes stay full although only half of the slots carry a block, and nothing outside this kernel has to compact the list.
    // Which thread sums which block depends on the flags alone, never on the batch size.
    const long long n3 = FR ? s1 : WB ? (long long)counts[1] : (pk.sel ? pk.n_sel_mp : lm.max_blocks);
    const long long po = (long long)prob * lm.slot_stride;  // the 3-D walk is in problem-local slots
    const uint8_t *flag3d = lm.flag3d + po, *type3d = lm.type3d + po;
    const double *geo3d = lm.geo3d + po * 9;
    __shared__ int q3[kLinThreads / 32][64];
    const int lane3 = threadIdx.x & 31, warp3 = threadIdx.x >> 5;
    int qlen = 0;                                                    // warp-uniform
    long long base = FR ? s0 : (long long)blockIdx.x * kLinThreads + warp3 * 32;  // first slot of this warp's next round
    for (long long it = t0;; it += stride) {
        long long slot = it;
        if (WB) {
            if (it >= n3) break;
            slot = lm.idx3d[it];
        } else {
            const bool more = base < n3;
            if (more) {
                const long long sl = base + lane3;
                const int rs = !FR && pk.sel && sl < n3 ? sel_slot(pk, (int)sl) : (int)sl;
                const bool on = sl < n3 && flag3d[rs];
                const unsigned mask = __ballot_sync(0xffffffffu, on);
                if (on) q3[warp3][qlen + __popc(mask & ((1u << lane3) - 1))] = rs;
                qlen += __popc(mask);
                base += stride;
                __syncwarp();
            }
            if (qlen < 32 && more) continue;      // keep collecting
            if (qlen == 0) break;                  // nothing left anywhere
            const int take = qlen < 32 ? qlen : 32;
            const int mine = lane3 < take ? q3[warp3][lane3] : -1;
            const int rest = lane3 + 32 < qlen ? q3[warp3][lane3 + 32] : 0;
            __syncwarp();
            if (lane3 + 32 < qlen) q3[warp3][lane3] = rest;
            qlen -= take;
            __syncwarp();
            if (mine < 0) continue;
            slot = mine;
        }
        const int type = type3d[slot];
        const LmCand &cb = reread(c);
        const double (*Wb)[7] = reread(W);
        double g[9], d[3];
#pragma unroll
        for (int i = 0; i < 9; ++i) g[i] = geo3d[slot * 9 + i];
        p3_values(cb, g, d);
        double rho0, sr;
        if (type == 1) {
            huber((d[0] * d[0] + d[1] * d[1]) + d[2] * d[2], pr.delta3d, rho0, sr);
            const long long blk = (long long)n2d + it;
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                const Row7 e = p3_point_row(cb, Wb, g, d, i);
                accumulate(A, e, sr);
                if (WB) put_row(bo, blk, i, e);
            }
            A.v[37] += 1.0;
            A.v[39] += 3.0;
            if (WB) put_head(bo, blk, 1, lm.slot_kf[po + slot], lm.slot_kp[po + slot], 3);
        } else {
            const Row7 e = p3_plane_row(cb, Wb, g, d);
            huber(e.a * e.a, pr.delta3d, rho0, sr);
            accumulate(A, e, sr);
            A.v[38] += 1.0;
            A.v[39] += 1.0;
            if (WB) {
                const long long blk = (long long)n2d + it;
                put_row(bo, blk, 0, e);
                put_head(bo, blk, 2, lm.slot_kf[po + slot], lm.slot_kp[po + slot], 1);
            }
        }
        A.v[0] += 0.5 * rho0;
    }

    // ---- CTA reduction (fixed order); FR: the warp's row
    __shared__ double red[kLinThreads / 32][kLinVals];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < kLinVals; ++i) {
        double x = A.v[i];
        for (int o = 16; o; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
        if (FR) {
            if (lane == 0) partial[((long long)blockIdx.y * partial_stride + fpos) * kLinVals + i] = x;
        } else if (lane == 0) {
            red[warp][i] = x;
        }
    }
    if (FR) return;
    __syncthreads();
    if (threadIdx.x < kLinVals) {
        double x = 0.0;
        for (int w = 0; w < kLinThreads / 32; ++w) x += red[w][threadIdx.x];
        partial[((long long)blockIdx.y * partial_stride + blockIdx.x) * kLinVals + threadIdx.x] = x;
    }
}


// ------------------------------------------------------------------ K4b': IBA_GPRFactor blocks
// IBACalib2.hpp:472-507 + TGPR::fit_predict (GPR.hpp:449-491): the neighbours are projected with the
// CURRENT extrinsic, K = sigma^2 exp(-D/2l^2) + sigma_n I, alpha = K^-1 y (Eigen::LLT), z = k*^T alpha,
// the keypoint is back-projected at depth z and re-projected into the covisible keyframes.
//
// K is conditioned like 1e12 (sigma_n = 1e-10), so HOW the derivative is formed decides its low digits.
// The reference differentiates by running the whole algorithm on ceres::Jet numbers; this kernel does the
// same, operation for operation: the kernel matrix, the unblocked lower Cholesky (Eigen's LLT for n < 32),
// both triangular solves and the prediction are evaluated on D7 duals in the order of the reference's
// loops (an adjoint formulation — one factorisation, no dual matrices — was measured 2e-6 off in J^T J,
// above the 1e-6 bar).  What can still differ from a CPU evaluation is exp() (<= 1 ulp between libms).
// One warp per block, lane i <-> row i; the dual matrix lives in shared memory, component-major, lower
// triangle packed.
constexpr int kGprTri = 32 * 33 / 2;
struct GprSmem {
    double L[8][kGprTri];                      // K, then its Cholesky factor (lower triangle, packed by rows)
    double xu[8][32], xv[8][32], y[8][32];     // neighbour pixels and depths (duals)
    double al[8][32];                          // alpha
};

__device__ __forceinline__ int tri(int i, int j) { return i * (i + 1) / 2 + j; }
__device__ __forceinline__ D7 ld7(const double (*m)[kGprTri], int idx) {
    D7 r; r.a = m[0][idx];
#pragma unroll
    for (int c = 0; c < 7; ++c) r.v[c] = m[1 + c][idx];
    return r;
}
__device__ __forceinline__ void st7(double (*m)[kGprTri], int idx, const D7 &x) {
    m[0][idx] = x.a;
#pragma unroll
    for (int c = 0; c < 7; ++c) m[1 + c][idx] = x.v[c];
}
__device__ __forceinline__ D7 ld7v(const double (*m)[32], int i) {
    D7 r; r.a = m[0][i];
#pragma unroll
    for (int c = 0; c < 7; ++c) r.v[c] = m[1 + c][i];
    return r;
}
__device__ __forceinline__ void st7v(double (*m)[32], int i, const D7 &x) {
    m[0][i] = x.a;
#pragma unroll
    for (int c = 0; c < 7; ++c) m[1 + c][i] = x.v[c];
}
__device__ __forceinline__ D7 d7_sqrt_dev(const D7 &f) {  // Jet sqrt: (sqrt a, f.v / (2 sqrt a))
    D7 r; r.a = sqrt(f.a);
    const double t = 1.0 / (2.0 * r.a);
#pragma unroll
    for (int c = 0; c < 7; ++c) r.v[c] = t * f.v[c];
    return r;
}
__device__ __forceinline__ D7 d7_exp_dev(const D7 &f) {   // Jet exp: (e^a, e^a f.v)
    D7 r; r.a = exp(f.a);
#pragma unroll
    for (int c = 0; c < 7; ++c) r.v[c] = r.a * f.v[c];
    return r;
}
__device__ __forceinline__ D7 shfl7(const D7 &x, int src) {
    D7 r; r.a = __shfl_sync(0xffffffffu, x.a, src);
#pragma unroll
    for (int c = 0; c < 7; ++c) r.v[c] = __shfl_sync(0xffffffffu, x.v[c], src);
    return r;
}

// grid (chunks, B), one warp per CTA.  FR (stl_linearize_frames): grid (n_sel, B), CTA x walks, in list order, the run of
// selection position x's keyframe in the problem's GPR list and writes its row at partial[blockIdx.y][x] (partial_stride = n_sel,
// partial_off = 0): the row's sum order depends on that keyframe's blocks alone.
template <bool WB, bool FR = false>
__global__ void __launch_bounds__(32)
k_linearize_gpr(const DevPack pk, const DevParams pr, const LmState lm, const LmCand *__restrict__ cands, const int *__restrict__ cprob,
                double *__restrict__ partial, int partial_stride, int partial_off, const BlockOut bo) {
    __shared__ GprSmem S;
    __shared__ LmCand c;
    __shared__ int list0;
    const int lane = threadIdx.x;
    const int prob = cprob ? cprob[blockIdx.y] : 0;
    {
        const double *src = reinterpret_cast<const double *>(cands + blockIdx.y);
        double *dst = reinterpret_cast<double *>(&c);
        for (int i = lane; i < (int)(sizeof(LmCand) / 8); i += 32) dst[i] = src[i];
    }
    lm_list_start(lm, prob, 3, &list0);
    __syncwarp();
    const int *counts = lm.d_counts + prob * 4;
    Acc A;
#pragma unroll
    for (int i = 0; i < kLinVals; ++i) A.v[i] = 0.0;
    const int C = pk.n_covis;
    const int nG = counts[3];
    int it0 = blockIdx.x, it1 = nG, step = gridDim.x;
    if (FR) {  // the keyframe's slots [mp_off, mp_off + n_mp) of problem prob
        const DevKf &Kf = pk.kf[sel_kf(pk, blockIdx.x)];
        const long long po = (long long)prob * lm.slot_stride;
        it0 = lower_pos(lm.idxG + list0, nG, po + Kf.mp_off);
        it1 = lower_pos(lm.idxG + list0, nG, po + Kf.mp_off + Kf.n_mp);
        step = 1;
    }
    for (int it = it0; it < it1; it += step) {
        const int cs = lm.idxG[list0 + it];  // global slot
        const int f = lm.slot_kf[cs];
        const uint32_t kp = lm.slot_kp[cs];
        const long long gblk = (long long)counts[0] + counts[1] + it;  // block index in stl_eval_blocks order
        const long long ms = cs;
        const int n = lm.gpr_m[ms];
        const DevKf &K = pk.kf[f];
        const double fx = K.fx, fy = K.fy, cx = K.cx, cy = K.cy;
        const float2 kxy = pk.kp_xy[K.kp_off + kp];
        const double u0 = kxy.x, v0 = kxy.y;
        // hyper-parameters of this factor (fitted per factor when params.gpr_optimize, IBACalib2.hpp:460-461); constants
        // as the reference forms them on Jets with zero partials: sigma*sigma, T(-0.5)/(l*l) = -0.5 * (1/(l*l))
        const double sigma = lm.gpr_hyper ? lm.gpr_hyper[ms * 2] : pr.gpr_sigma, ell = lm.gpr_hyper ? lm.gpr_hyper[ms * 2 + 1] : pr.gpr_l;
        const double sigma2 = sigma * sigma;
        const double inv_l2 = 1.0 / (ell * ell);
        const double coef = -0.5 * inv_l2;
        const D7 kdiag = d7_const(sigma2 * exp(coef * 0.0) + pr.gpr_noise);
        __syncwarp();
        // 1. neighbour j -> camera frame with the candidate, pixel coordinates X_j and depth y_j (IBACalib2.hpp:478-489)
        D7 myu = d7_const(0.0), myv = d7_const(0.0);
        if (lane < n) {
            const uint32_t p = lm.gpr_nb[ms * kMaxK + lane];
            const double px = (double)pk.px[K.pt_off + p], py = (double)pk.py[K.pt_off + p], pz = (double)pk.pz[K.pt_off + p];
            D7 tf[3];
#pragma unroll
            for (int i = 0; i < 3; ++i) tf[i] = ((c.R[i * 3] * px + c.R[i * 3 + 1] * py) + c.R[i * 3 + 2] * pz) + c.t[i];
            myu = (tf[0] * fx) / tf[2] + cx;
            myv = (tf[1] * fy) / tf[2] + cy;
            st7v(S.xu, lane, myu); st7v(S.xv, lane, myv); st7v(S.y, lane, tf[2]);
        }
        __syncwarp();
        // 2. kernel matrix, lower triangle: K(i, j) = sigma2 * exp(coef * |X_j - X_i|^2) for j < i (self_pdist, GPR.hpp:41-54,
        //    forms it at (ri = j, ci = i) as d = X[ri] - X[ci] and mirrors it); diagonal sigma2 * exp(0) + sigma_noise
        if (lane < n) {
            for (int j = 0; j < lane; ++j) {
                const D7 dx = ld7v(S.xu, j) - myu, dy = ld7v(S.xv, j) - myv;
                const D7 kv = d7_exp_dev((dx * dx + dy * dy) * coef) * sigma2;
                st7(S.L, tri(lane, j), kv);
            }
            st7(S.L, tri(lane, lane), kdiag);
        }
        __syncwarp();
        // 3. Eigen::LLT, unblocked (n < 32): for k: L_kk = sqrt(K_kk - sum_j L_kj^2); L_ik = (K_ik - sum_j L_ij L_kj) / L_kk
        for (int k = 0; k < n; ++k) {
            D7 v = d7_const(0.0);
            if (lane >= k && lane < n) {
                v = ld7(S.L, tri(lane, k));
                for (int j = 0; j < k; ++j) v = v - ld7(S.L, tri(lane, j)) * ld7(S.L, tri(k, j));
            }
            D7 xk = shfl7(v, k);
            xk = d7_sqrt_dev(xk);
            if (lane == k) st7(S.L, tri(k, k), xk);
            else if (lane > k && lane < n) st7(S.L, tri(lane, k), v / xk);
            __syncwarp();
        }
        // 4. alpha = K^-1 y: forward substitution (row order), then backward (each row sums its terms in ascending column order)
        {
            D7 v = lane < n ? ld7v(S.y, lane) : d7_const(0.0);
            for (int j = 0; j < n; ++j) {
                D7 aj = v / ld7(S.L, tri(min(lane, n - 1), min(lane, n - 1)));  // meaningful on lane j only
                aj = shfl7(aj, j);
                if (lane == j) v = aj;
                else if (lane > j && lane < n) v = v - ld7(S.L, tri(lane, j)) * aj;
            }
            if (lane < n) st7v(S.al, lane, v);
            __syncwarp();
            for (int i = n - 1; i >= 0; --i) {
                if (lane == i) {
                    D7 w = ld7v(S.al, i);
                    for (int j = i + 1; j < n; ++j) w = w - ld7(S.L, tri(j, i)) * ld7v(S.al, j);
                    st7v(S.al, i, w / ld7(S.L, tri(i, i)));
                }
                __syncwarp();
            }
        }
        // 5. Kstar_j = sigma2 * exp((-0.5 * inv_l2) * |X_j - x*|^2) (rbf_kernel_2d, GPR.hpp:57-63), z = sum_j Kstar_j alpha_j in j order
        D7 term = d7_const(0.0);
        if (lane < n) {
            const D7 dx = myu - u0, dy = myv - v0;
            const D7 ks = d7_exp_dev((dx * dx + dy * dy) * (-0.5 * inv_l2)) * sigma2;
            term = ks * ld7v(S.al, lane);
        }
        D7 z = d7_const(0.0);
        for (int j = 0; j < n; ++j) z = z + shfl7(term, j);
        // 6. back-projection at depth z, covisible re-projection, Huber, normal equations (lane 0)
        if (lane == 0) {
            const double ifx = 1.0 / fx, ify = 1.0 / fy;  // Jet division by a constant: multiply by 1/g
            const D7 P0[3] = {(z * (u0 - cx)) * ifx, (z * (v0 - cy)) * ify, z};
            double sq = 0.0;
            int nres = 0;
            for (int s = 0; s < C; ++s) {
                if (!pk.covis_valid[f * C + s]) continue;
                const float2 uv = pk.covis_uv[(K.kp_off + kp) * C + s];
                if (isnan(uv.x)) continue;
                const float *rp = pk.relpose + ((long long)f * C + s) * 12;
                double P1[3];
                for (int i = 0; i < 3; ++i)
                    P1[i] = (((double)rp[i * 4] * P0[0].a + (double)rp[i * 4 + 1] * P0[1].a) + (double)rp[i * 4 + 2] * P0[2].a) + (double)rp[i * 4 + 3] * c.s.a;
                const double eu = (fx * P1[0] / P1[2] + cx) - (double)uv.x, ev = (fy * P1[1] / P1[2] + cy) - (double)uv.y;
                sq += eu * eu;
                sq += ev * ev;
                nres += 2;
            }
            double rho0, sr;
            huber(sq, pr.delta2d, rho0, sr);
            A.v[0] += 0.5 * rho0;
            A.v[40] += 1.0;
            A.v[39] += (double)nres;
            int wrow = 0;
            for (int s = 0; s < C; ++s) {
                if (!pk.covis_valid[f * C + s]) continue;
                const float2 uv = pk.covis_uv[(K.kp_off + kp) * C + s];
                if (isnan(uv.x)) continue;
                const float *rp = pk.relpose + ((long long)f * C + s) * 12;
                D7 P1[3];
                for (int i = 0; i < 3; ++i)
                    P1[i] = ((P0[0] * (double)rp[i * 4] + P0[1] * (double)rp[i * 4 + 1]) + P0[2] * (double)rp[i * 4 + 2]) + c.s * (double)rp[i * 4 + 3];
                const D7 eu = ((P1[0] * fx) / P1[2] + cx) - (double)uv.x;
                const D7 ev = ((P1[1] * fy) / P1[2] + cy) - (double)uv.y;
                accumulate(A, eu, sr);
                accumulate(A, ev, sr);
                if (WB) { put_row(bo, gblk, wrow, eu); put_row(bo, gblk, wrow + 1, ev); wrow += 2; }
            }
            if (WB) put_head(bo, gblk, 3, f, kp, nres);
        }
    }
    // per-CTA partial: lane 0 holds the sums
    __shared__ double red[kLinVals];
    if (lane == 0)
        for (int i = 0; i < kLinVals; ++i) red[i] = A.v[i];
    __syncwarp();
    for (int i = lane; i < kLinVals; i += 32)
        partial[((long long)blockIdx.y * partial_stride + partial_off + blockIdx.x) * kLinVals + i] = red[i];
}

// Position in the kLinVals packed sums (cost, g[7], the upper triangle of H by rows, counts) of value v of the STL_LIN_NSUMS
// record (cost, g[7], H[7][7] full, counts)
__device__ __forceinline__ int lin_packed(int v) {
    if (v < 8) return v;
    if (v >= 57) return v - 21;
    const int i = (v - 8) / 7, j = (v - 8) % 7, a = i < j ? i : j, b = i < j ? j : i;
    return 8 + a * 7 - a * (a - 1) / 2 + (b - a);
}

// one CTA per candidate: sums the per-CTA partials in order and expands H to the full symmetric 7x7
// one CTA of 1024 threads per candidate: warp w sums values w, w+32 over the chunks (lane-strided partial
// sums, then a shuffle tree: a fixed order, so the result is reproducible)
__global__ void __launch_bounds__(1024)
k_lin_finish(const double *__restrict__ partial, int nchunks, double *__restrict__ out, int out_stride, const P2pView P) {
    __shared__ double tot[kLinVals];
    const int b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int v = warp; v < kLinVals; v += 32) {
        double x = 0.0;
        for (int i = lane; i < nchunks; i += 32) x += partial[((long long)b * nchunks + i) * kLinVals + v];
        for (int o = 16; o; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
        if (lane == 0) tot[v] = x;
    }
    __syncthreads();
    if (threadIdx.x < STL_LIN_NSUMS) out[(long long)b * out_stride + threadIdx.x] = tot[lin_packed(threadIdx.x)];
    if (P.n > 1) p2p_allreduce_record(P, b, out + (long long)b * out_stride + P.off);  // keyframes sharded over GPUs: sum the shards here
}

// per-keyframe rows: one thread per value of out[b][sel_kf(pos)][STL_LIN_NSUMS] = plane / point row + GPR row (in that order)
__global__ void k_lin_frames_finish(const DevPack pk, const double *__restrict__ rows, const double *__restrict__ rows_gpr, int B,
                                    double *__restrict__ out /*[B][n_kf][STL_LIN_NSUMS]*/) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)B * pk.n_sel * STL_LIN_NSUMS) return;
    const int v = (int)(i % STL_LIN_NSUMS);
    const long long r = i / STL_LIN_NSUMS;  // b * n_sel + pos
    const int b = (int)(r / pk.n_sel), pos = (int)(r % pk.n_sel);
    const long long src = r * kLinVals + lin_packed(v);
    out[((long long)b * pk.n_kf + sel_kf(pk, pos)) * STL_LIN_NSUMS + v] = rows_gpr ? rows[src] + rows_gpr[src] : rows[src];
}

template <class T> void dfree(T *&p) { if (p) { cudaFree(p); p = nullptr; } }

}  // namespace

void lm_free(LmState &lm) {
    dfree(lm.slot_kf); dfree(lm.slot_kp); dfree(lm.flags); dfree(lm.geo2d); dfree(lm.geo3d);
    dfree(lm.idxG); dfree(lm.gpr_nb); dfree(lm.gpr_m); dfree(lm.gpr_hyper);
    dfree(lm.amap); dfree(lm.stage); dfree(lm.plane_a); dfree(lm.nnb_pos); dfree(lm.nbb); dfree(lm.nbbx); dfree(lm.nbb_m); dfree(lm.nbb_last);
    dfree(lm.idx2d); dfree(lm.idx3d); dfree(lm.d_sel); dfree(lm.d_tmp); dfree(lm.partial); dfree(lm.frames); dfree(lm.d_cand);
    if (lm.h_cand) cudaFreeHost(lm.h_cand);
    if (lm.h_counts) cudaFreeHost(lm.h_counts);
    if (lm.h_amap) cudaFreeHost(lm.h_amap);
    delete[] lm.n_blocks;
    if (lm.h2d_done) cudaEventDestroy(lm.h2d_done);
    if (lm.counts_done) cudaEventDestroy(lm.counts_done);
    if (lm.amap_done) cudaEventDestroy(lm.amap_done);
    lm = LmState();
}

// The buffers of a set of P problems with `lanes` association lanes (sized by the pack): allocated by the first association, or
// ahead of it by a caller that wants LmState::nnb_pos / nbb_m filled by K2a.  The per-problem arrays and the lane scratch are
// high-water marks: reallocated only when more problems / lanes are asked for than they hold (a driver that alternates single
// steps and sets pays no allocation per switch); a failure frees everything (no half-built set).
cudaError_t lm_reserve(const DevPack &pk, const DevParams &pr, LmState &lm, int P, int lanes, cudaStream_t st) {
    cudaError_t e;
#define TRY(x) do { e = (x); if (e != cudaSuccess) { lm_free(lm); return e; } } while (0)
    // block slots = query slots: one per map-point-carrying keypoint (a twelfth of the keypoints at the KITTI-00 shape), so the
    // flag arrays the selects compact, and the per-block geometry, are that much smaller than one-per-keypoint arrays
    const long long ns = pk.n_mp_total > 0 ? pk.n_mp_total : 1;
    if (lm.n_slots != ns || lm.P_cap < P) {
        lm_free(lm);  // P_cap stays 0 until every allocation below succeeded: a failure midway starts over next time
        const long long nsa = (ns + 15) / 16 * 16, n = nsa * P;
        lm.slot_stride = nsa;
        TRY(cudaMalloc(&lm.slot_kf, 4 * n)); TRY(cudaMalloc(&lm.slot_kp, 4 * n));
        // the four per-slot flag arrays and the counters are one allocation: one memset per new set
        lm.flags_bytes = (size_t)(4 * n + 16 * P);
        TRY(cudaMalloc(&lm.flags, lm.flags_bytes));
        lm.flag2d = lm.flags; lm.type3d = lm.flags + n; lm.flag3d = lm.flags + 2 * n; lm.flagG = lm.flags + 3 * n;
        lm.d_counts = reinterpret_cast<int *>(lm.flags + 4 * n);
        TRY(cudaMalloc(&lm.geo2d, 48 * n)); TRY(cudaMalloc(&lm.geo3d, 72 * n));
        TRY(cudaMalloc(&lm.idx2d, 4 * n)); TRY(cudaMalloc(&lm.idx3d, 4 * ns)); TRY(cudaMalloc(&lm.idxG, 4 * n));
        if (pr.use_gpr) { TRY(cudaMalloc(&lm.gpr_nb, 4 * n * kMaxK)); TRY(cudaMalloc(&lm.gpr_m, 4 * n)); }
        TRY(cudaMalloc(&lm.d_sel, 8));
        size_t tb = 0;
        cub::CountingInputIterator<int> it(0);
        TRY(cub::DeviceSelect::Flagged(nullptr, tb, it, lm.flag2d, lm.idx2d, lm.d_sel, (int)n, st));
        lm.tmp_bytes = tb;
        TRY(cudaMalloc(&lm.d_tmp, tb));
        TRY(cudaMallocHost(&lm.h_counts, 16 * (size_t)P));
        lm.n_blocks = new long long[4 * (size_t)P]();
        TRY(cudaEventCreateWithFlags(&lm.counts_done, cudaEventDisableTiming));
        TRY(cudaEventCreateWithFlags(&lm.amap_done, cudaEventDisableTiming));
        lm.n_slots = ns;
        lm.max_blocks = ns;
        lm.P_cap = P;
    }
    if (lanes > lm.lane_cap) {
        dfree(lm.amap); dfree(lm.stage); dfree(lm.plane_a); dfree(lm.nnb_pos); dfree(lm.nbb); dfree(lm.nbbx); dfree(lm.nbb_m); dfree(lm.nbb_last);
        if (lm.h_amap) cudaFreeHost(lm.h_amap);
        lm.h_amap = nullptr;
        lm.lane_cap = 0;
        const long long nm = ns * lanes;
        TRY(cudaMalloc(&lm.amap, sizeof(int2) * lanes)); TRY(cudaMallocHost(&lm.h_amap, sizeof(int2) * lanes));
        TRY(cudaMalloc(&lm.stage, nm)); TRY(cudaMalloc(&lm.plane_a, 32 * nm)); TRY(cudaMalloc(&lm.nnb_pos, 4 * nm));
        TRY(cudaMalloc(&lm.nbb, 4 * nm * kMaxK)); TRY(cudaMalloc(&lm.nbbx, sizeof(float4) * nm * kMaxK)); lm.nbbx_stride = nm;
        TRY(cudaMalloc(&lm.nbb_m, 4 * nm)); TRY(cudaMalloc(&lm.nbb_last, 8 * nm));
        lm.lane_cap = lanes;
        // the single association's lane: workspace slot 0, problem 0 (what K2a's folded 1-NN assumes); lm_set_lanes skips the
        // copy while the first lane stays what h_amap[0] says is on the device
        lm.h_amap[0] = make_int2(0, 0);
        TRY(cudaMemcpy(lm.amap, lm.h_amap, sizeof(int2), cudaMemcpyHostToDevice));
    }
#undef TRY
    return cudaSuccess;
}

cudaError_t lm_begin(const DevPack &pk, const DevParams &pr, LmState &lm, int P, bool partial, int lanes, cudaStream_t st) {
    cudaError_t e = lm_reserve(pk, pr, lm, P, lanes, st);
    if (e != cudaSuccess) return e;
    lm.ready = false;
    lm.clear_lanes = partial;
    if (!partial) {  // the flag arrays of a set of P are packed for P (the allocation holds P_cap): one memset of what P uses
        const long long n = lm.slot_stride * P;
        lm.P = P;
        lm.flag2d = lm.flags; lm.type3d = lm.flags + n; lm.flag3d = lm.flags + 2 * n; lm.flagG = lm.flags + 3 * n;
        lm.d_counts = reinterpret_cast<int *>(lm.flags + 4 * n);
        e = cudaMemsetAsync(lm.flags, 0, (size_t)(4 * n + 16 * P), st);
    }
    return e;
}

cudaError_t lm_set_lanes(LmState &lm, const int2 *lanes, int n, cudaStream_t st) {
    if (n > lm.lane_cap) return cudaErrorInvalidValue;
    lm.lane0 = lanes[0];
    if (n == 1 && lanes[0].x == lm.h_amap[0].x && lanes[0].y == lm.h_amap[0].y) return cudaSuccess;  // already on the device
    cudaError_t e = cudaEventSynchronize(lm.amap_done);
    if (e != cudaSuccess) return e;
    memcpy(lm.h_amap, lanes, sizeof(int2) * n);
    e = cudaMemcpyAsync(lm.amap, lm.h_amap, sizeof(int2) * n, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaEventRecord(lm.amap_done, st);
    return e;
}

// Enqueues BuildProblem of n lanes on `st` and returns without waiting: the block counts stay on the device (d_counts: plane,
// 3-D, point-to-point, GPR per problem), where the linearisation kernels read them; lm_copy_counts puts a copy in pinned host
// memory behind `counts_done` for callers that want the numbers (lm_block_counts).
cudaError_t lm_associate(const DevPack &pk, const DevWork &wk, const DevParams &pr, LmState &lm, int n, cudaStream_t st, bool hints, bool cert,
                         int part, bool nn_folded) {
    cudaError_t e;
#define TRY(x) do { e = (x); if (e != cudaSuccess) return e; } while (0)
    const dim3 grid((unsigned)(pk.n_sel * wk.sub), (unsigned)n);  // selection positions: unselected keyframes keep the cleared flags
    if (part != 2) {
        lm.ready = false;
        lm.sub = wk.sub;
        if (lm.clear_lanes) k_lm_clear<<<dim3((unsigned)((lm.slot_stride + 1023) / 1024 < 64 ? (lm.slot_stride + 1023) / 1024 : 64), (unsigned)n), 256, 0, st>>>(lm);
        if (pk.n_sel > 0) {
            if (!(pr.plane_index && !pr.use_gpr))  // with the plane index there is no neighbourhood to search at the scan point
                k_lm_knn_a<<<grid, kWarps * 32, 0, st>>>(pk, wk, pr, lm);
            k_lm_plane_a<<<grid, 128, 0, st>>>(pk, wk, pr, lm);
        }
        TRY(cudaGetLastError());
    }
    if (part == 1 || pk.n_sel == 0) return cudaSuccess;  // an empty selection: no blocks
    if (!nn_folded) k_lm_knn_b<<<grid, kWarps * 32, 0, st>>>(pk, wk, pr, lm, hints, cert);  // else K2a has filled nnb_pos / nbb_m
    k_lm_plane_b<<<grid, 128, 0, st>>>(pk, wk, pr, lm);
    TRY(cudaGetLastError());
#undef TRY
    return cudaSuccess;
}

// the 3-D/2-D blocks are complete after k_lm_plane_a: their dense list (the linearisation walks it) needs nothing of the 3-D
// search.  ONE select over the flags of all P problems: each problem's run comes out in slot order, and a problem that was not
// re-associated gets back exactly the run it had
cudaError_t lm_compact2d(LmState &lm, cudaStream_t st) {
    cub::CountingInputIterator<int> it(0);
    size_t tb = lm.tmp_bytes;
    return cub::DeviceSelect::Flagged(lm.d_tmp, tb, it, lm.flag2d, lm.idx2d, lm.d_sel, (int)(lm.slot_stride * lm.P), st);
}

cudaError_t lm_finish_associate(LmState &lm, bool use_gpr, cudaStream_t st) {
    // the 3-D/3-D blocks are counted by k_lm_plane_b and walked slot by slot by the linearisation: their dense list is only
    // built for stl_eval_blocks (lm_compact3d)
    lm.idx3d_valid = false;
    if (use_gpr) {
        cub::CountingInputIterator<int> it(0);
        size_t tb = lm.tmp_bytes;
        const cudaError_t e = cub::DeviceSelect::Flagged(lm.d_tmp, tb, it, lm.flagG, lm.idxG, lm.d_sel + 1, (int)(lm.slot_stride * lm.P), st);
        if (e != cudaSuccess) return e;
    }
    lm.counts_valid = false;
    lm.use_gpr = use_gpr;
    lm.clear_lanes = false;
    lm.ready = true;
    return cudaSuccess;
}

// Dense list of the 3-D/3-D blocks of problem 0 (slot order), for the numbered walk of stl_eval_blocks.
cudaError_t lm_compact3d(const DevPack &pk, LmState &lm, cudaStream_t st) {
    if (lm.idx3d_valid) return cudaSuccess;
    const long long ns = pk.n_mp_total > 0 ? pk.n_mp_total : 1;
    cub::CountingInputIterator<int> it(0);
    size_t tb = lm.tmp_bytes;
    const cudaError_t e = cub::DeviceSelect::Flagged(lm.d_tmp, tb, it, lm.flag3d, lm.idx3d, lm.d_counts + 1, (int)ns, st);
    if (e == cudaSuccess) lm.idx3d_valid = true;
    return e;
}

// The read-back of the block counts of every problem of the set.
cudaError_t lm_copy_counts(LmState &lm, cudaStream_t st) {
    cudaError_t e = cudaMemcpyAsync(lm.h_counts, lm.d_counts, 16 * (size_t)lm.P, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaEventRecord(lm.counts_done, st);
    return e;
}

// Host copy of the block counts of the last association (waits for it to finish).
cudaError_t lm_block_counts(LmState &lm) {
    if (!lm.ready) return cudaErrorNotReady;
    if (lm.counts_valid) return cudaSuccess;
    cudaError_t e = cudaEventSynchronize(lm.counts_done);
    if (e != cudaSuccess) return e;
    for (int p = 0; p < lm.P; ++p) {
        const int *h = lm.h_counts + 4 * p;
        long long *o = lm.n_blocks + 4 * p;
        o[0] = h[0]; o[1] = h[2]; o[2] = h[1] - h[2]; o[3] = lm.use_gpr ? h[3] : 0;
    }
    lm.counts_valid = true;
    return cudaSuccess;
}

namespace {
// training data of GPR::fit for GPR block `it` of a problem (list run from l0, nG blocks): neighbour j -> (u, v, depth) with the
// association extrinsic (IBACalib2.hpp:449-457: pt = R p + t; uv = fx pt0 / pt2 + cx, fy pt1 / pt2 + cy), fp64, one thread per neighbour
__global__ void k_gpr_train(const DevPack pk, const DevCand *__restrict__ c0, const LmState lm, int l0, double *__restrict__ out /*[nG][32][3]*/,
                            int *__restrict__ out_n) {
    const int it = blockIdx.x, lane = threadIdx.x;
    const long long ms = lm.idxG[l0 + it];  // global slot
    const int f = lm.slot_kf[ms];
    const int n = lm.gpr_m[ms];
    const DevKf &K = pk.kf[f];
    const DevCand &c = *c0;
    if (lane == 0) out_n[it] = n;
    double u = 0, v = 0, z = 0;
    if (lane < n) {
        const uint32_t p = lm.gpr_nb[ms * kMaxK + lane];
        double X, Y, Z;
        xform(c.R, c.t, (double)pk.px[K.pt_off + p], (double)pk.py[K.pt_off + p], (double)pk.pz[K.pt_off + p], X, Y, Z);
        u = (double)K.fx * X / Z + (double)K.cx;
        v = (double)K.fy * Y / Z + (double)K.cy;
        z = Z;
    }
    double *o = out + ((long long)it * kMaxK + lane) * 3;
    o[0] = u; o[1] = v; o[2] = z;
}
__global__ void k_gpr_scatter_hyper(const LmState lm, int l0, int nG, const double *__restrict__ fitted /*[nG][2]*/, double *__restrict__ hyper) {
    const int it = blockIdx.x * blockDim.x + threadIdx.x;
    if (it >= nG) return;
    const long long ms = lm.idxG[l0 + it];
    hyper[ms * 2] = fitted[it * 2];
    hyper[ms * 2 + 1] = fitted[it * 2 + 1];
}
__global__ void k_gpr_gather_hyper(const LmState lm, const DevParams pr, int nG, double *__restrict__ out /*[nG][2]*/) {
    const int it = blockIdx.x * blockDim.x + threadIdx.x;
    if (it >= nG) return;
    const long long ms = lm.idxG[it];  // problem 0: its run starts the list
    out[it * 2] = lm.gpr_hyper ? lm.gpr_hyper[ms * 2] : pr.gpr_sigma;
    out[it * 2 + 1] = lm.gpr_hyper ? lm.gpr_hyper[ms * 2 + 1] : pr.gpr_l;
}
}  // namespace

cudaError_t lm_fit_gpr_hyper(const DevPack &pk, const DevCand *c0, const DevParams &pr, LmState &lm, int prob, cudaStream_t st, int flavour) {
    cudaError_t e = lm_block_counts(lm);
    if (e != cudaSuccess) return e;
    const int nG = (int)lm.n_blocks[4 * prob + 3];
    int l0 = 0;
    for (int q = 0; q < prob; ++q) l0 += (int)lm.n_blocks[4 * q + 3];
    if (!lm.gpr_hyper) {
        e = cudaMalloc(&lm.gpr_hyper, 16 * lm.slot_stride * lm.P_cap);
        if (e != cudaSuccess) return e;
    }
    if (nG == 0) return cudaSuccess;
    double *d_train = nullptr, *d_fit = nullptr;
    int *d_n = nullptr;
    std::vector<double> h_train((size_t)nG * kMaxK * 3), h_fit((size_t)nG * 2);
    std::vector<int> h_n(nG);
    e = cudaMalloc(&d_train, 8 * h_train.size());
    if (e == cudaSuccess) e = cudaMalloc(&d_n, 4 * (size_t)nG);
    if (e == cudaSuccess) e = cudaMalloc(&d_fit, 16 * (size_t)nG);
    if (e == cudaSuccess) {
        k_gpr_train<<<nG, kMaxK, 0, st>>>(pk, c0, lm, l0, d_train, d_n);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(h_train.data(), d_train, 8 * h_train.size(), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(h_n.data(), d_n, 4 * (size_t)nG, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) {
#pragma omp parallel for schedule(dynamic, 16)
        for (int it = 0; it < nG; ++it) {
            const int n = h_n[it];
            double x[kMaxK * 2], y[kMaxK];
            for (int j = 0; j < n; ++j) {
                x[j * 2] = h_train[((size_t)it * kMaxK + j) * 3];
                x[j * 2 + 1] = h_train[((size_t)it * kMaxK + j) * 3 + 1];
                y[j] = h_train[((size_t)it * kMaxK + j) * 3 + 2];
            }
            const GprFitResult r = gpr_fit(x, y, n, pr.gpr_noise, pr.gpr_sigma, pr.gpr_l, 15, flavour);  // max_num_iterations = 15 (GPR.hpp:360)
            h_fit[(size_t)it * 2] = r.sigma;
            h_fit[(size_t)it * 2 + 1] = r.l;
        }
        e = cudaMemcpyAsync(d_fit, h_fit.data(), 16 * (size_t)nG, cudaMemcpyHostToDevice, st);
    }
    if (e == cudaSuccess) {
        k_gpr_scatter_hyper<<<(nG + 127) / 128, 128, 0, st>>>(lm, l0, nG, d_fit, lm.gpr_hyper);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(d_train); cudaFree(d_n); cudaFree(d_fit);
    return e;
}

cudaError_t lm_get_gpr_hyper(const DevParams &pr, LmState &lm, double *out, cudaStream_t st) {
    cudaError_t e = lm_block_counts(lm);
    const int nG = (int)lm.n_blocks[3];
    if (e != cudaSuccess || nG == 0) return e;
    double *d = nullptr;
    e = cudaMalloc(&d, 16 * (size_t)nG);
    if (e != cudaSuccess) return e;
    k_gpr_gather_hyper<<<(nG + 127) / 128, 128, 0, st>>>(lm, pr, nG, d);
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, d, 16 * (size_t)nG, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(d);
    return e;
}

// Sim3Exp / SE3Exp duals of the B parameter vectors and the problem of each, host -> device: the first thing lm_linearize
// does, or — ahead of it — a caller that has other work to put on the stream in between (the overlapped step)
cudaError_t lm_stage_candidates(LmState &lm, const double *x, const int *problem, int B, cudaStream_t st) {
    cudaError_t e;
#define TRY(x) do { e = (x); if (e != cudaSuccess) return e; } while (0)
    const size_t bytes = (sizeof(LmCand) + sizeof(int)) * (size_t)B;
    if (B > lm.cand_cap) {
        dfree(lm.d_cand);
        if (lm.h_cand) cudaFreeHost(lm.h_cand);
        lm.h_cand = nullptr;
        lm.cand_cap = 0;
        TRY(cudaMalloc(&lm.d_cand, bytes));
        TRY(cudaMallocHost(&lm.h_cand, bytes));
        lm.cand_cap = B;
    }
    LmCand *hc = reinterpret_cast<LmCand *>(lm.h_cand);
    int *hp = reinterpret_cast<int *>(hc + B);
    if (!lm.h2d_done) TRY(cudaEventCreateWithFlags(&lm.h2d_done, cudaEventDisableTiming));
    TRY(cudaEventSynchronize(lm.h2d_done));
    for (int b = 0; b < B; ++b) { make_lm_candidate(x + (size_t)b * 7, hc + b); hp[b] = problem ? problem[b] : 0; }
    TRY(cudaMemcpyAsync(lm.d_cand, hc, bytes, cudaMemcpyHostToDevice, st));
    TRY(cudaEventRecord(lm.h2d_done, st));
#undef TRY
    return cudaSuccess;
}

cudaError_t lm_linearize(const DevPack &pk, const DevParams &pr, LmState &lm, const double *x, const int *problem, int B, double *d_out,
                         cudaStream_t st, const BlockOut *blocks, int out_stride, const P2pView *p2p, cudaEvent_t before_finish, bool cand_staged) {
    cudaError_t e;
#define TRY(x) do { e = (x); if (e != cudaSuccess) return e; } while (0)
    if (!cand_staged) TRY(lm_stage_candidates(lm, x, problem, B, st));
    const LmCand *cands = reinterpret_cast<const LmCand *>(lm.d_cand);
    // the staged problem index is read only when the caller named problems (stl_*_multi)
    const int *cprob = problem ? reinterpret_cast<const int *>(cands + B) : nullptr;
    // grids are sized from the host-side upper bound of the block count (one block per map-point-carrying
    // keypoint at most) — never from the counts themselves, so that the chunking, and with it the order
    // of the fp64 sums, is the same whether or not the host has looked at the counts; the kernels read
    // the exact counts from the device
    const long long work = pk.sel ? (pk.n_sel_mp > 0 ? pk.n_sel_mp : 1) : lm.max_blocks;  // a selection: what a pack of it would have
    long long chunks_ll = (work + kLinThreads * 2 - 1) / (kLinThreads * 2);
    // at most ONE wave of CTAs per candidate at 2 CTAs per SM: 296 chunks measured 0.134 ms against 0.140 (592), 0.163 (444: a
    // wave and a half) and 0.157 (1184) at the KITTI-00 shape, and the finishing kernel sums four times fewer partials.  444 chunks at
    // 3 CTAs per SM take 0.853 ms per step against 0.869 (296 at 2 CTAs per SM), but the chunk count sets the order of the fp64
    // sums: changing it changes the cost's last bits
    static const int kChunkCap = getenv("STL_LIN_CHUNKS") ? atoi(getenv("STL_LIN_CHUNKS")) : 148 * 2;
    int chunks = (int)(chunks_ll < 1 ? 1 : (chunks_ll > kChunkCap ? kChunkCap : chunks_ll));
    const long long gwork = lm.use_gpr ? work : 0;
    long long gchunks_ll = gwork > 0 ? (gwork + 3) / 4 : 0;
    int gchunks = (int)(gchunks_ll > 148 * 8 ? 148 * 8 : gchunks_ll);
    const int stride = chunks + gchunks;
    const long long need = (long long)B * stride * kLinVals;
    if (need > lm.partial_cap) {
        dfree(lm.partial);
        TRY(cudaMalloc(&lm.partial, 8 * need));
        lm.partial_cap = need;
    }
    const BlockOut bo = blocks ? *blocks : BlockOut();
    if (blocks) {
        TRY(lm_compact3d(pk, lm, st));
        k_linearize<true, 1><<<dim3(chunks, B), kLinThreads, 0, st>>>(pk, pr, lm, cands, cprob, lm.partial, stride, bo);
    } else if ((long long)chunks * B <= 148 * 2) {
        // one candidate (the step): one wave at two CTAs per SM, which a third CTA slot would leave unused; unbounded, the
        // kernel takes 222 registers without spills (0.114 against 0.120 ms at 168 registers with 128 B of spills)
        k_linearize<false, 1><<<dim3(chunks, B), kLinThreads, 0, st>>>(pk, pr, lm, cands, cprob, lm.partial, stride, bo);
    } else {
        // a batch (the poll): several waves, three CTAs per SM at 168 registers (13.7 ms per 256-candidate poll against 14.0
        // at four CTAs per SM)
        k_linearize<false, 3><<<dim3(chunks, B), kLinThreads, 0, st>>>(pk, pr, lm, cands, cprob, lm.partial, stride, bo);
    }
    TRY(cudaGetLastError());
    if (gchunks > 0) {
        if (blocks) k_linearize_gpr<true><<<dim3(gchunks, B), 32, 0, st>>>(pk, pr, lm, cands, cprob, lm.partial, stride, chunks, bo);
        else k_linearize_gpr<false><<<dim3(gchunks, B), 32, 0, st>>>(pk, pr, lm, cands, cprob, lm.partial, stride, chunks, bo);
        TRY(cudaGetLastError());
    }
    if (before_finish) TRY(cudaStreamWaitEvent(st, before_finish, 0));
    k_lin_finish<<<B, 1024, 0, st>>>(lm.partial, stride, d_out, out_stride > 0 ? out_stride : STL_LIN_NSUMS, p2p ? *p2p : P2pView());
    TRY(cudaGetLastError());
#undef TRY
    return cudaSuccess;
}

// Per-keyframe rows of B candidates (stl_linearize_frames): the plane / point rows (k_linearize<false, 1, true>), the GPR rows
// (k_linearize_gpr<false, true>), then k_lin_frames_finish adds them and scatters them into the zeroed [B][n_kf][STL_LIN_NSUMS]
// output in lm.frames, returned in *d_out.  No exchange: the rows are this context's keyframes.
cudaError_t lm_linearize_frames(const DevPack &pk, const DevParams &pr, LmState &lm, const double *x, const int *problem, int B, double **d_out,
                                cudaStream_t st) {
    cudaError_t e;
#define TRY(x) do { e = (x); if (e != cudaSuccess) return e; } while (0)
    TRY(lm_stage_candidates(lm, x, problem, B, st));
    const LmCand *cands = reinterpret_cast<const LmCand *>(lm.d_cand);
    const int *cprob = problem ? reinterpret_cast<const int *>(cands + B) : nullptr;
    const long long nrow = (long long)B * pk.n_sel, nout = (long long)B * pk.n_kf * STL_LIN_NSUMS;
    const long long need = nrow * kLinVals * (lm.use_gpr ? 2 : 1) + nout;  // 8 (41 + 41 use_gpr + 62) bytes per (candidate, keyframe)
    if (need > lm.frames_cap) {
        dfree(lm.frames);
        lm.frames_cap = 0;
        TRY(cudaMalloc(&lm.frames, 8 * need));
        lm.frames_cap = need;
    }
    double *rows = lm.frames, *rows_gpr = lm.use_gpr ? rows + nrow * kLinVals : nullptr;
    double *out = lm.frames + nrow * kLinVals * (lm.use_gpr ? 2 : 1);
    *d_out = out;
    if (pk.sel || pk.n_sel < pk.n_kf) TRY(cudaMemsetAsync(out, 0, 8 * (size_t)nout, st));  // rows of unselected keyframes
    if (pk.n_sel == 0) return cudaSuccess;
    const int fw = kLinThreads / 32;  // keyframes per CTA
    k_linearize<false, 1, true><<<dim3((unsigned)((pk.n_sel + fw - 1) / fw), (unsigned)B), kLinThreads, 0, st>>>(pk, pr, lm, cands, cprob, rows, pk.n_sel, BlockOut());
    TRY(cudaGetLastError());
    if (rows_gpr) {
        k_linearize_gpr<false, true><<<dim3((unsigned)pk.n_sel, (unsigned)B), 32, 0, st>>>(pk, pr, lm, cands, cprob, rows_gpr, pk.n_sel, 0, BlockOut());
        TRY(cudaGetLastError());
    }
    const long long nv = nrow * STL_LIN_NSUMS;
    k_lin_frames_finish<<<(unsigned)((nv + 255) / 256), 256, 0, st>>>(pk, rows, rows_gpr, B, out);
    TRY(cudaGetLastError());
#undef TRY
    return cudaSuccess;
}

}  // namespace stl
