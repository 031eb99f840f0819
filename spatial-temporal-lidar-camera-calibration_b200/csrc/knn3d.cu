// knn3d.cu — K2: 3-D/3-D alignment term of BAError.
//
// Replaces, per 2-D correspondence that carries a map point:
//   map point -> LiDAR frame        src/examples/iba_global.cpp:231-234
//   ComputeAlignmentDist            src/examples/iba_global.cpp:111-156
//     (1-NN :116-121, k-NN of the neighbour :125-129, radius truncation :130-133,
//      gates :136-139, ComputeCovariance + FastEigen3x3_EV :140-143, regression
//      gate and point-to-plane / point-to-point distance :144-154)
//   thresholded accumulation        src/examples/iba_global.cpp:239-251
//
// Two kernels, so that each stays small enough for the instruction cache and uses the
// machine the way its work is shaped (profiles/r01_k2_*.txt):
//   K2a k_nn_knn     one WARP per query: exact 1-NN, then exact k-NN around that neighbour;
//                    writes the neighbour list (sorted positions, distance order).
//   K2b k_plane_dist one THREAD per query: gates, ordered covariance, closed-form eigenvector,
//                    regression gate, distance; fixed-order CTA reduction per (candidate, keyframe).
// plus the stand-alone k-NN entry used by the parity tests.
#include <algorithm>
#include <cstdlib>

#include "kernels.h"
#include "knn.cuh"

namespace stl {
namespace {

constexpr int kWarps = 8;
#ifndef STL_KNN_MINB
#define STL_KNN_MINB 8  // resident CTAs per SM the traversal kernels are compiled for (32 registers, full occupancy; measured best of 4..8)
#endif
constexpr int kPlaneThreads = 128;
#ifndef STL_PLANE_MINB
#define STL_PLANE_MINB 5  // 96 registers: measured 4 / 5 / 6 / 8 -> 119 / 106 / 131 / 126 us for k_plane_dist
#endif

// the map point of correspondence `kp` in the LiDAR frame of candidate c (iba_global.cpp:231-234)
__device__ __forceinline__ void map_point_lidar(const DevPack &pk, const DevKf &K, const DevCand &c, int f, uint32_t kp, double &qx,
                                                double &qy, double &qz) {
    const float *Tcw = pk.Tcw + (long long)f * 12;
    const float *mp = pk.kp_mp + (K.kp_off + kp) * 3;
    // GetWorldPos()*scale evaluated in float32, then widened (iba_global.cpp:232; SURVEY.md A6)
    const double wx = (double)__fmul_rn(mp[0], c.sf), wy = (double)__fmul_rn(mp[1], c.sf), wz = (double)__fmul_rn(mp[2], c.sf);
    // TcwRS = Tcw with the translation scaled (iba_global.cpp:206-208)
    const double cxm = dadd(dot3e((double)Tcw[0], (double)Tcw[1], (double)Tcw[2], wx, wy, wz), dmul((double)Tcw[3], c.s));
    const double cym = dadd(dot3e((double)Tcw[4], (double)Tcw[5], (double)Tcw[6], wx, wy, wz), dmul((double)Tcw[7], c.s));
    const double czm = dadd(dot3e((double)Tcw[8], (double)Tcw[9], (double)Tcw[10], wx, wy, wz), dmul((double)Tcw[11], c.s));
    xform(c.Ri, c.ti, cxm, cym, czm, qx, qy, qz);  // Tcl.inverse() * P
}

// K2a — grid: (candidate, keyframe, sub-block).  A warp draws `batch` queries at a time: everything that is a function of ONE
// query (the map point in the LiDAR frame, the seed distance at the associated scan point, the distance to the home box — 40 %
// of the kernel's instructions when every lane repeats them for the same query) is computed one query per LANE, then the warp
// searches the queries one after another with those scalars broadcast.
__global__ void __launch_bounds__(kWarps * 32, STL_KNN_MINB)
k_nn_knn(const DevPack pk, const DevWork wk, const DevParams pr, const int B, const int batch, uint32_t *__restrict__ lm_pos,
         int *__restrict__ lm_m) {
    const int sub = wk.sub;
    const int j = blockIdx.x % sub;
    const int bf = blockIdx.x / sub;
    const int fi = bf / B, f = sel_kf(pk, fi), b = bf - fi * B;
    const int nq = wk.n_q[(long long)b * pk.n_kf + f];
    if (nq <= 0) return;
    const int lane = threadIdx.x & 31;
    const DevKf K = pk.kf[f];
    const DevCand &c = wk.cand[b];
    ScanView S = make_view(pk, K);
    S.stats = wk.dbg_stats;
    const long long cbase = (long long)b * pk.n_kp_total + K.kp_off;
    const long long qbase = (long long)b * pk.n_mp_total + K.mp_off;
    __shared__ int ticket;
    if (threadIdx.x == 0) ticket = 0;
    __syncthreads();
    for (;;) {
        const int t0 = next_ticket(&ticket, lane) * batch;
        if ((long long)t0 * sub + j >= nq) break;
        // ---- one query per lane
        const int qi = (t0 + lane) * sub + j;
        const bool valid = lane < batch && qi < nq;
        double qx = 0, qy = 0, qz = 0, sd = DBL_MAX;
        uint32_t hint = 0, soi = 0xffffffffu, spos = 0xffffffffu;
        float delta = 0.f;
        if (valid) {
            const uint2 ks = wk.q_kpsp[cbase + qi];  // (keypoint, associated scan position)
            hint = ks.y;
            map_point_lidar(pk, K, c, f, ks.x, qx, qy, qz);
            // Sink1::seed at the associated scan point
            const double dd = dist3e(qx, qy, qz, (double)S.px[hint], (double)S.py[hint], (double)S.pz[hint]);
            if (dd == dd) { sd = dd; soi = S.orig[hint]; spos = hint; }
            delta = home_box_delta(S, (int)(hint >> 5), qx, qy, qz);
        }
        uint32_t out_pos = 0xffffffffu;
        float out_g2 = 0.f;
        // ---- the warp searches them one after another
        unsigned todo = __ballot_sync(kFull, valid);
        while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            const double x = __shfl_sync(kFull, qx, src), y = __shfl_sync(kFull, qy, src), z = __shfl_sync(kFull, qz, src);
            const uint32_t h = __shfl_sync(kFull, hint, src);
            Sink1 nn;
            nn.d = __shfl_sync(kFull, sd, src);
            nn.oi = __shfl_sync(kFull, soi, src);
            nn.pos = __shfl_sync(kFull, spos, src);
            if (nn.pos != 0xffffffffu) nn.df = __double2float_ru(nn.d);
            nn_near_leaf_seeded(S, pr.adj_r, (int)(h >> 5), x, y, z, nn, lane, __shfl_sync(kFull, delta, src));
            if (lane == src) { out_pos = nn.pos; out_g2 = nn.g2; }
            if (pr.use_plane && !pr.plane_index) {  // with the plane index the neighbourhood of nn is already fitted
                const long long slot = qbase + (long long)(t0 + src) * sub + j;
                SinkK kn(pr.k, pr.radius2);
                knn_around_point(S, nn.pos, kn, lane);
                wk.nb[slot * kMaxK + lane] = lane < kn.count ? kn.kpos : 0xffffffffu;
                store_nb_coords(wk.nbx, wk.nbx_stride, slot, S, lane, kn.count, kn.kpos);
                const double last = __shfl_sync(kFull, kn.kd, kn.count > 0 ? kn.count - 1 : 0);
                if (lane == 0) { wk.nb_m[slot] = kn.count; wk.nb_last[slot] = last; }
            }
        }
        if (valid) { wk.nn_pos[qbase + qi] = out_pos; wk.nn_g2[qbase + qi] = out_g2; }
        // ---- one LM iteration at this extrinsic (stl_step_batch): BuildProblem asks for the 1-NN of the SAME map point scaled
        // in fp64 (q', iba_local.cpp:283), a few micrometres from q.  Everything k_lm_knn_b would gather again is in registers
        // here, so the question is settled on the spot — by the certificate (lm.cu: sqrt(g2) - |q - q'| > |q' - h|: every other
        // point is strictly farther from q' than h), else by an exact search seeded with h — and that kernel is not launched.
        if (lm_pos != nullptr && b == 0) {
            double lx = 0, ly = 0, lz = 0, nn_d = DBL_MAX;
            uint32_t nn_p = 0xffffffffu;
            bool need = false;
            if (valid) {
                const float *Tcw = pk.Tcw + (long long)f * 12;
                const float *mp = pk.kp_mp + (K.kp_off + wk.q_kpsp[cbase + qi].x) * 3;
                const double ma = (double)mp[0], mb = (double)mp[1], mc = (double)mp[2];
                const double Mx = dadd(dot3e((double)Tcw[0], (double)Tcw[1], (double)Tcw[2], ma, mb, mc), (double)Tcw[3]);
                const double My = dadd(dot3e((double)Tcw[4], (double)Tcw[5], (double)Tcw[6], ma, mb, mc), (double)Tcw[7]);
                const double Mz = dadd(dot3e((double)Tcw[8], (double)Tcw[9], (double)Tcw[10], ma, mb, mc), (double)Tcw[11]);
                xform(c.Ri, c.ti, dmul(Mx, c.s), dmul(My, c.s), dmul(Mz, c.s), lx, ly, lz);  // initSE3.inverse() * (MapPoint * init_scale)
                need = true;
                if (out_pos != 0xffffffffu) {
                    const double move = sqrt(dist3e(qx, qy, qz, lx, ly, lz)) * (1.0 + 1e-9) + 1e-12;  // |q - q'|, rounded up
                    const double dh = dist3e(lx, ly, lz, (double)S.px[out_pos], (double)S.py[out_pos], (double)S.pz[out_pos]);
                    const double reach = (double)__fsqrt_rd(out_g2) - move;                          // every other point is at least this far from q'
                    if (reach > 0.0 && reach * reach > dh * (1.0 + 1e-6) + 1e-18) { need = false; nn_p = out_pos; nn_d = dh; }
                }
            }
            unsigned todo2 = __ballot_sync(kFull, need);
            while (todo2) {
                const int src = __ffs(todo2) - 1;
                todo2 &= todo2 - 1;
                const double x = __shfl_sync(kFull, lx, src), y = __shfl_sync(kFull, ly, src), z = __shfl_sync(kFull, lz, src);
                uint32_t h = __shfl_sync(kFull, out_pos, src);
                if (h == 0xffffffffu) h = __shfl_sync(kFull, hint, src);
                Sink1 nn;
                nn_near_leaf(S, pr.adj_r, (int)(h >> 5), x, y, z, nn, lane, h);
                if (lane == src) { nn_p = nn.pos; nn_d = nn.d; }
            }
            if (valid) {
                const long long slot = K.mp_off + qi;
                if (nn_d > pr.max_3d_dist2) {  // iba_local.cpp:289
                    lm_pos[slot] = 0xffffffffu;
                } else {
                    lm_pos[slot] = nn_p;
                    lm_m[slot] = nn_p == hint ? -2 : -3;  // the associated scan point itself (its plane is known) / looked up by k_lm_plane_b
                }
            }
        }
    }
}

// K2b — grid: (candidate, keyframe, sub-block), one thread per query
__global__ void __launch_bounds__(kPlaneThreads, STL_PLANE_MINB)
k_plane_dist(const DevPack pk, const DevWork wk, const DevParams pr, const int B, const int debug) {
    const int sub = wk.sub;
    const int j = blockIdx.x % sub;
    const int bf = blockIdx.x / sub;
    const int fi = bf / B, f = sel_kf(pk, fi), b = bf - fi * B;
    const long long rec = (long long)b * pk.n_kf + f;
    const int nq = wk.n_q[rec];
    double s3d = 0, v3d = 0, c3d = 0, vpl = 0, vpt = 0;
    if (nq > 0) {
        const DevKf K = pk.kf[f];
        const DevCand &c = wk.cand[b];
        const ScanView S = make_view(pk, K);
        const long long cbase = (long long)b * pk.n_kp_total + K.kp_off;
        const long long qbase = (long long)b * pk.n_mp_total + K.mp_off;
        for (int qi = j * kPlaneThreads + threadIdx.x; qi < nq; qi += sub * kPlaneThreads) {
            const uint32_t kp = wk.corr_kp[cbase + wk.q_corr[cbase + qi]];
            double qx, qy, qz;
            map_point_lidar(pk, K, c, f, kp, qx, qy, qz);
            const uint32_t np = wk.nn_pos[qbase + qi];
            const double nx = (double)S.px[np], ny = (double)S.py[np], nz = (double)S.pz[np];
            const double dx = dsub(nx, qx), dy = dsub(ny, qy), dz = dsub(nz, qz);
            double dist = sqrt(dot3e(dx, dy, dz, dx, dy, dz));  // pt2pt (iba_global.cpp:122)
            int is_plane = 0, m = 0;
            if (pr.use_plane) {
                const PlaneOut po = pr.plane_index ? plane_lookup(pk, K, np)
                                                   : plane_fit(NbCoords{wk.nbx + qbase + qi, wk.nbx_stride}, wk.nb_m[qbase + qi], wk.nb_last[qbase + qi], nx, ny, nz, pr, pr.variant == 1);
                m = po.m;
                if (po.gates_ok && !(po.reg > pr.reg_thr)) {  // iba_global.cpp:147
                    is_plane = 1;
                    dist = fabs(dot3e(dx, dy, dz, po.n.x, po.n.y, po.n.z));
                }
            }
            if (dist < pr.thr3d) {  // iba_global.cpp:241-249
                s3d += dist; v3d += 1.0;
                if (is_plane) vpl += 1.0; else vpt += 1.0;
            }
            c3d += 1.0;
            if (debug) {
                const long long o = K.kp_off + qi;
                wk.dbg_nn[o] = S.orig[np];
                wk.dbg_m[o] = m;
                wk.dbg_plane[o] = is_plane;
                wk.dbg_dist[o] = dist;
                for (int t = 0; t < kMaxK; ++t) {
                    const uint32_t p = (pr.use_plane && !pr.plane_index && t < m) ? wk.nb[(qbase + qi) * kMaxK + t] : 0xffffffffu;
                    wk.dbg_knn[o * kMaxK + t] = p == 0xffffffffu ? 0xffffffffu : S.orig[p];
                }
            }
        }
    }
    // fixed-order CTA reduction
    __shared__ double red[5][kPlaneThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int o = 16; o; o >>= 1) {
        s3d += __shfl_down_sync(0xffffffffu, s3d, o); v3d += __shfl_down_sync(0xffffffffu, v3d, o);
        c3d += __shfl_down_sync(0xffffffffu, c3d, o); vpl += __shfl_down_sync(0xffffffffu, vpl, o);
        vpt += __shfl_down_sync(0xffffffffu, vpt, o);
    }
    if (lane == 0) { red[0][warp] = s3d; red[1][warp] = v3d; red[2][warp] = c3d; red[3][warp] = vpl; red[4][warp] = vpt; }
    __syncthreads();
    if (threadIdx.x == 0) {
        AlignRec r = {0, 0, 0, 0, 0};
        for (int w = 0; w < kPlaneThreads / 32; ++w) { r.s3d += red[0][w]; r.v3d += red[1][w]; r.c3d += red[2][w]; r.vpl += red[3][w]; r.vpt += red[4][w]; }
        wk.align[rec * sub + j] = r;
    }
}

// stand-alone exact k-NN: one warp per query
__global__ void __launch_bounds__(kWarps * 32)
k_knn3d(const DevPack pk, const int kf, const double *__restrict__ q, const int nq, const int k, const double radius2,
        uint32_t *__restrict__ out_idx, double *__restrict__ out_d2, int *__restrict__ out_cnt) {
    const int lane = threadIdx.x & 31;
    const int qi = blockIdx.x * kWarps + (threadIdx.x >> 5);
    if (qi >= nq) return;
    const DevKf K = pk.kf[kf];
    const ScanView S = make_view(pk, K);
    SinkK kn(k, radius2 > 0 ? radius2 : DBL_MAX);
    traverse(S, q[qi * 3], q[qi * 3 + 1], q[qi * 3 + 2], kn, lane);
    if (lane < k) {
        out_idx[(long long)qi * k + lane] = lane < kn.count ? kn.ki : 0xffffffffu;
        out_d2[(long long)qi * k + lane] = lane < kn.count ? kn.kd : INFINITY;
    }
    if (lane == 0) out_cnt[qi] = kn.count;
}

// ---- plane index: local plane of every scan point, computed once per pack ---------------------
// grid (blocks, nkf): one warp per point of the keyframe range; lists go to a scratch buffer
__global__ void __launch_bounds__(kWarps * 32, STL_KNN_MINB)
k_index_knn(const DevPack pk, const int kf_begin, const DevParams pr, const long long first_pt, uint32_t *__restrict__ nb,
            int *__restrict__ nb_m, double *__restrict__ nb_last) {
    const DevKf K = pk.kf[kf_begin + blockIdx.y];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const ScanView S = make_view(pk, K);
    for (int p = blockIdx.x * kWarps + warp; p < K.n_pts; p += gridDim.x * kWarps) {
        SinkK kn(pr.k, pr.radius2);
        knn_around_point(S, (uint32_t)p, kn, lane);
        const long long o = K.pt_off - first_pt + p;
        nb[o * kMaxK + lane] = lane < kn.count ? kn.kpos : 0xffffffffu;
        const double last = __shfl_sync(kFull, kn.kd, kn.count > 0 ? kn.count - 1 : 0);
        if (lane == 0) { nb_m[o] = kn.count; nb_last[o] = last; }
    }
}

__global__ void __launch_bounds__(kPlaneThreads)
k_index_plane(const DevPack pk, const int kf_begin, const DevParams pr, const long long first_pt, const uint32_t *__restrict__ nb,
              const int *__restrict__ nb_m, const double *__restrict__ nb_last) {
    const DevKf K = pk.kf[kf_begin + blockIdx.y];
    const ScanView S = make_view(pk, K);
    for (int p = blockIdx.x * kPlaneThreads + threadIdx.x; p < K.n_pad; p += gridDim.x * kPlaneThreads) {
        PlaneRec r = {0.0, 0.0, 0.0, 0.0};
        int mm = -1;
        if (p < K.n_pts) {
            const long long o = K.pt_off - first_pt + p;
            const PlaneOut po = plane_thread(S, nb + o * kMaxK, nb_m[o], nb_last[o], (double)S.px[p], (double)S.py[p], (double)S.pz[p], pr, pr.variant == 1);
            r.nx = po.n.x; r.ny = po.n.y; r.nz = po.n.z; r.reg = po.reg;
            mm = po.gates_ok ? po.m : -(po.m + 1);
        }
        pk.pl_rec[K.pt_off + p] = r;
        pk.pl_m[K.pt_off + p] = mm;
    }
}

}  // namespace

cudaError_t build_plane_index(const DevPack &pk, const DevKf *h_kf, int kf_begin, int nkf, const DevParams &pr, cudaStream_t st,
                              BuildScratch &scr) {
    const long long first = h_kf[kf_begin].pt_off;
    const long long npts = h_kf[kf_begin + nkf - 1].pt_off + h_kf[kf_begin + nkf - 1].n_pad - first;
    if (npts <= 0) return cudaSuccess;
    int max_pts = 0;
    for (int f = 0; f < nkf; ++f) max_pts = max_pts > h_kf[kf_begin + f].n_pad ? max_pts : h_kf[kf_begin + f].n_pad;
    cudaError_t e = scr.need(2, 4 * (size_t)npts * kMaxK);
    if (e == cudaSuccess) e = scr.need(4, 4 * (size_t)npts);
    if (e == cudaSuccess) e = scr.need(3, 8 * (size_t)npts);
    if (e != cudaSuccess) return e;
    uint32_t *nb = (uint32_t *)scr.buf[2]; int *m = (int *)scr.buf[4]; double *last = (double *)scr.buf[3];
    const int bx = (max_pts + kWarps * 16 - 1) / (kWarps * 16);  // ~16 points per warp
    k_index_knn<<<dim3(bx, nkf), kWarps * 32, 0, st>>>(pk, kf_begin, pr, first, nb, m, last);
    k_index_plane<<<dim3((max_pts + kPlaneThreads * 4 - 1) / (kPlaneThreads * 4), nkf), kPlaneThreads, 0, st>>>(pk, kf_begin, pr, first, nb, m, last);
    return cudaGetLastError();  // stream order protects the scratch: the next chunk's kernels run after these
}

namespace {
__global__ void k_debug_trig(const double *__restrict__ x, int n, double *__restrict__ ac, double *__restrict__ co) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    ac[i] = acos_cr(fmin(fmax(x[i], -1.0), 1.0));
    co[i] = cos_cr(x[i]);
}
}  // namespace

cudaError_t launch_debug_trig(const double *d_x, int n, double *d_acos, double *d_cos, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    k_debug_trig<<<(n + 255) / 256, 256, 0, st>>>(d_x, n, d_acos, d_cos);
    return cudaGetLastError();
}

cudaError_t launch_align3d(const DevPack &pk, const DevWork &wk, const DevParams &pr, int B, int debug, cudaStream_t st, cudaEvent_t after_traversal,
                           uint32_t *lm_pos, int *lm_m) {
    if (B <= 0) return cudaSuccess;
    if (pk.n_sel <= 0) return after_traversal ? cudaEventRecord(after_traversal, st) : cudaSuccess;
    // queries a warp draws at a time: the per-query preamble runs one query per lane, the searches one after another — a long
    // batch is cheap in instructions and long in latency, so small keyframe shards or selections (one wave of CTAs) get the short one
    int batch = (long long)pk.n_sel * B >= 600 ? 8 : 4;
    if (const char *e = getenv("STL_K2_BATCH")) batch = std::max(1, std::min(32, atoi(e)));
    k_nn_knn<<<(unsigned)(pk.n_sel * B * wk.sub), kWarps * 32, 0, st>>>(pk, wk, pr, B, batch, lm_pos, lm_m);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    if (after_traversal && (e = cudaEventRecord(after_traversal, st)) != cudaSuccess) return e;
    k_plane_dist<<<(unsigned)(pk.n_sel * B * wk.sub), kPlaneThreads, 0, st>>>(pk, wk, pr, B, debug);
    return cudaGetLastError();
}

cudaError_t launch_knn3d(const DevPack &pk, int kf, const double *d_q, int nq, int k, double radius2, uint32_t *d_idx, double *d_d2,
                         int *d_cnt, cudaStream_t st) {
    if (nq <= 0) return cudaSuccess;
    k_knn3d<<<(nq + kWarps - 1) / kWarps, kWarps * 32, 0, st>>>(pk, kf, d_q, nq, k, radius2, d_idx, d_d2, d_cnt);
    return cudaGetLastError();
}

}  // namespace stl
