// assoc2d.cu — K1: transform + project + 2-D association + 3-D/2-D and hand-eye terms.
//
// Replaces, per (candidate, keyframe):
//   TransformPointCloud            include/pointcloud.h:82-86   (iba_global.cpp:199)
//   FindProjectCorrespondences     src/examples/iba_global.cpp:55-96
//     (projection + cull :68-81, KDTree2D build :84, 1-NN per keypoint :85-95)
//   frame gate                     src/examples/iba_global.cpp:203
//   hand-eye term                  src/examples/iba_global.cpp:264-276
//   covisible re-projection term   src/examples/iba_global.cpp:291-328
//
// PERSISTENT: two CTAs per SM draw (keyframe, candidate) units from a global ticket; a unit is worked by one CTA from its
// keypoint tables (ONE cp.async.bulk per keyframe, mbarrier completion) to its FrameRec.  No index is ever built over the projected points (the
// reference rebuilds a KD-tree per candidate and keyframe): only points within max_pixel_dist
// of a keypoint can become a correspondence, so the scan is STREAMED (SoA float4, 12 B/point)
// through a float32 pre-cull against a shared-memory occupancy bitmap of the dilated keypoints.
// The scan is KD-ordered (K0), so whole cells that cannot project into the image are skipped
// from their bounding boxes without being loaded.  The ~2 % survivors are re-evaluated in the
// reference's exact fp64 arithmetic against the keypoints of their 8 px grid cells (grid and
// keypoints staged in shared memory) and min-reduced per keypoint with (distance, original
// index) order — the KD-tree 1-NN + threshold whenever no exact distance tie exists.  A survivor is
// recorded with its coordinates in an L2-resident per-CTA list, so nothing after the stream gathers
// from the scan.  Bound: HBM for the stream, instruction latency for the survivor phases (DESIGN.md §K1).
#include <algorithm>
#include <mutex>

#include "kernels.h"
#include "se3.cuh"

namespace stl {
namespace {

constexpr int kThreads = 512;
constexpr int kSurvCap = kK1SurvCap;
constexpr int kMatchCap = kK1MatchCap;  // (keypoint, point) matches a unit may record between the two exact passes
constexpr unsigned long long kInf64 = 0x7ff0000000000000ull;  // +inf bits
constexpr unsigned long long kNoKey = 0xffffffffffffffffull;
static_assert(kSurvCap <= 4096, "a correspondence key keeps the survivor slot in 12 bits");

struct Smem {  // fixed part; dynamic arrays follow
    float mu[4], mv[4], mz[4];  // fast projection rows: u*z, v*z, z
    float zmin, ub_u, ub_v, ez;
    float u_hi, v_hi;
    float4 plane[5];   // conservative half-spaces of "may pass the pre-cull": a.xyz . p + a.w >= thr
    float thr[5];
    int n_surv, overflow, n_groups, n_match, next_group;
    // persistent-loop state (written by thread 0 between two barriers, read by everybody)
    int unit, u_end, new_tab, cur_f;
    int next_ticket, have_next;  // drawn ahead by a helper thread while the current unit runs
    int n_cells;                 // visible level-1 cells of the current unit
    unsigned covis_mask;  // bit j: covisible slot j of this keyframe is valid
    double he_val;
    int warp_cnt[16], warp_q[16];
    int base_corr, base_q;
    double red[3][16];
    unsigned long long mbar;  // completion of the table blob's bulk copy
};

// ---- bulk copy global -> shared with mbarrier completion (cp.async.bulk, SASS UBLKCP) ------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src, uint32_t bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// earlier generic-proxy accesses of shared memory are ordered before the async-proxy write that follows
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void bulk_prefetch_l2(const void *src, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}

template <bool STABLE>
__device__ __forceinline__ bool exact_project(const DevCand &c, double fx, double cx, double cy, double W, double H, float xf,
                                              float yf, float zf, double &u, double &v) {
    double xc, yc, zc;
    xform(c.R, c.t, (double)xf, (double)yf, (double)zf, xc, yc, zc);
    if (!(zc > 0.0)) return false;
    u = ddiv(dadd(dmul(fx, xc), dmul(cx, zc)), zc);
    v = ddiv(dadd(dmul(fx, yc), dmul(cy, zc)), zc);  // fx, not fy (iba_global.cpp:73)
    if (STABLE) {  // iba_global_stable.cpp:92-94: the rounded pixel (half away from zero) must be inside
        const double ru = round(u), rv = round(v);
        return (0.0 <= ru && ru < W && 0.0 <= rv && rv < H);
    }
    return (0.0 <= u && u < W && 0.0 <= v && v < H);
}

// hand-eye term ||log(Tcl*Tl) - log(Tc*Tcl)|| of one keyframe (iba_global.cpp:264-276); kept out of
// line so that its 4x4 temporaries do not inflate the streaming kernel's register budget
__device__ __noinline__ double hand_eye_term(const DevPack &pk, const DevCand &c, int f) {
    double TcR[9], Tct[3], TlR[9], Tlt[3], C1R[9], C1t[3], C2R[9], C2t[3], l1[6], l2[6];
    const float *tc = pk.he_Tc + (long long)f * 12;
    const double *tl = pk.he_Tl + (long long)f * 12;
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) { TcR[i * 3 + j] = (double)tc[i * 4 + j]; TlR[i * 3 + j] = tl[i * 4 + j]; }
        Tct[i] = dmul((double)tc[i * 4 + 3], c.s);  // Tc.topRightCorner *= scale
        Tlt[i] = tl[i * 4 + 3];
    }
    rt_compose(c.R, c.t, TlR, Tlt, C1R, C1t);
    rt_compose(TcR, Tct, c.R, c.t, C2R, C2t);
    se3_log(C1R, C1t, l1);
    se3_log(C2R, C2t, l2);
    double ss = 0;
    for (int i = 0; i < 6; ++i) { const double d = l1[i] - l2[i]; ss += d * d; }
    return sqrt(ss);
}

// Can any point of the box satisfy all five half-spaces?  max over the box of a.p + w is
// a.c + |a|.e + w (c = centre, e = half extent); float32 evaluation error is covered by a relative
// slack of 2^-16 on the magnitude of the terms.  Empty boxes (lo > hi) are never visible.
__device__ __forceinline__ bool box_visible(const Smem &S, float4 lo, float4 hi) {
    if (!(lo.x <= hi.x)) return false;
    const float cx = 0.5f * (lo.x + hi.x), cy = 0.5f * (lo.y + hi.y), cz = 0.5f * (lo.z + hi.z);
    const float ex = 0.5f * (hi.x - lo.x), ey = 0.5f * (hi.y - lo.y), ez = 0.5f * (hi.z - lo.z);
    bool vis = true;
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        const float4 a = S.plane[i];
        const float ax = fabsf(a.x), ay = fabsf(a.y), az = fabsf(a.z);
        const float spread = fmaf(ax, ex, fmaf(ay, ey, az * ez));
        const float centre = fmaf(a.x, cx, fmaf(a.y, cy, fmaf(a.z, cz, a.w)));
        const float mag = fmaf(ax, fabsf(cx), fmaf(ay, fabsf(cy), fmaf(az, fabsf(cz), fabsf(a.w)))) + spread;
        vis = vis && (centre + spread + 1.52587890625e-05f * mag >= S.thr[i]);
    }
    return vis;
}

// shared-memory views of the per-keyframe tables
struct Tables {
    unsigned long long *best_d2, *best_key;  // [n_kp]
    // views into the keyframe's table blob (common.cuh: K1Tab), brought in by one bulk copy
    const float2 *kp;                        // [n_kp]
    const uint32_t *bm;                      // bitmap
    const unsigned short *gstart, *gkp;      // [gw*gh+1], [n_kp]
    const uint32_t *has_mp;                  // [(n_kp+31)/32]
    unsigned short *groups;                  // [n_pad/128]
    unsigned short *cells;                   // [n_pad/1024] visible level-1 cells
};

// A correspondence key: (original index << 32) | (sorted position << 12) | survivor slot.  Original indices are unique
// within a scan, so the minimum over keys is the minimum over original indices; position (< 2^20) and slot (< 2^12) ride along.
__device__ __forceinline__ uint32_t key_low(uint32_t si, uint32_t slot) { return (si << 12) | slot; }

// Exact fp64 evaluation of one surviving scan point against the keypoints around its projection.
// PASS 1: atomicMin of the squared distance per keypoint, appending every match to the unit's list;
// PASS 2 (only when that list overflowed): ties -> atomicMin of (original index, position).
template <int PASS>
__device__ __forceinline__ void exact_point(const DevPack &pk, const DevKf &K, const DevCand &c, const DevParams &pr, const Tables &T,
                                            float xf, float yf, float zf, uint32_t si, uint32_t slot, ulonglong2 *matches, int *n_match) {
    double u, v;
    const bool stable = pk.kp_xyd != nullptr;
    if (stable ? !exact_project<true>(c, (double)K.fx, (double)K.cx, (double)K.cy, (double)K.W, (double)K.H, xf, yf, zf, u, v)
               : !exact_project<false>(c, (double)K.fx, (double)K.cx, (double)K.cy, (double)K.W, (double)K.H, xf, yf, zf, u, v)) return;
    const double rp = sqrt(pr.max_pixel_dist2) + (stable ? 1e-3 : 1e-6);  // stable: cells are keyed by the float32 copy
    int gx0 = (int)floor((u - rp) * (1.0 / kGridCell)), gx1 = (int)floor((u + rp) * (1.0 / kGridCell));
    int gy0 = (int)floor((v - rp) * (1.0 / kGridCell)), gy1 = (int)floor((v + rp) * (1.0 / kGridCell));
    gx0 = max(gx0, 0); gy0 = max(gy0, 0); gx1 = min(gx1, K.gw - 1); gy1 = min(gy1, K.gh - 1);
    for (int gy = gy0; gy <= gy1; ++gy) {
        const int a = T.gstart[gy * K.gw + gx0], b = T.gstart[gy * K.gw + gx1 + 1];  // cells of one row are contiguous
        for (int j = a; j < b; ++j) {
            const int k = T.gkp[j];
            double qx, qy;
            if (stable) { const double2 q = pk.kp_xyd[K.kp_off + k]; qx = q.x; qy = q.y; }
            else { const float2 q = T.kp[k]; qx = (double)q.x; qy = (double)q.y; }
            const double dx = dsub(qx, u), dy = dsub(qy, v);
            const double d2 = dadd(dmul(dx, dx), dmul(dy, dy));  // nanoflann.hpp:524-535, query - data
            if (d2 <= pr.max_pixel_dist2) {
                const unsigned long long bits = (unsigned long long)__double_as_longlong(d2);
                if (PASS == 1) {
                    atomicMin(&T.best_d2[k], bits);
                    const int m = atomicAdd(n_match, 1);  // remembered for the tie pass (coalesced list in L2)
                    if (m < kMatchCap) matches[m] = make_ulonglong2(bits, ((unsigned long long)k << 32) | key_low(si, slot));
                } else if (bits == T.best_d2[k]) {
                    atomicMin(&T.best_key[k], ((unsigned long long)pk.orig[K.pt_off + si] << 32) | key_low(si, slot));
                }
            }
        }
    }
}

// PERSISTENT: gridDim.x CTAs (two per SM) draw chunks of `chunk` consecutive (keyframe, candidate) units from a global
// ticket; consecutive units of a chunk share the keyframe when B > 1, so the table blob stays in shared memory.
__global__ void __launch_bounds__(kThreads, 2)
k_assoc2d(const DevPack pk, const DevWork wk, const DevParams pr, const int B, const int with_terms, const int n_units, const int chunk,
          const int max_kp, const int max_tab, const int max_groups) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem &S = *reinterpret_cast<Smem *>(smem_raw);
    unsigned char *const tab = smem_raw + ((sizeof(Smem) + 15) & ~size_t(15));
    Tables T;
    {
        unsigned char *q = tab + max_tab;
        T.best_d2 = reinterpret_cast<unsigned long long *>(q); q += 8 * (size_t)max_kp;
        T.best_key = reinterpret_cast<unsigned long long *>(q); q += 8 * (size_t)max_kp;
        T.groups = reinterpret_cast<unsigned short *>(q); q += 2 * (size_t)max_groups;
        T.cells = reinterpret_cast<unsigned short *>(q);
    }
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        mbar_init(&S.mbar, 1);
        S.unit = -1; S.u_end = 0; S.cur_f = -1; S.new_tab = 0; S.have_next = 0;
    }
    uint32_t tab_phase = 0;
    for (;;) {
    __syncthreads();  // the previous unit is finished by every thread: tables, records and S are free again
    long long clk_top = 0;
    if (wk.k1_clk != nullptr && tid == 0) clk_top = clock64();
    // ---- prologue, thread 0: next unit (from the chunk in hand or a new ticket), table blob on its way (one bulk copy),
    // fast rows, error bounds, culling half-spaces.  Everybody else clears the per-keypoint minima meanwhile.
    if (tid == 0) {
        int u = S.unit + 1;
        if (S.unit < 0 || u >= S.u_end) {
            const long long t0 = (long long)(S.have_next ? S.next_ticket : atomicAdd(wk.k1_ticket, 1)) * chunk;
            S.have_next = 0;
            if (t0 >= n_units) {  // every CTA draws exactly one failing ticket; the last one to leave re-arms the counters
                if (atomicAdd(wk.k1_ticket + 1, 1) == (int)gridDim.x - 1) { wk.k1_ticket[0] = 0; wk.k1_ticket[1] = 0; __threadfence(); }
                u = -1;
            } else {
                u = (int)t0;
                S.u_end = (int)min(t0 + chunk, (long long)n_units);
            }
        }
        S.unit = u;
        if (u >= 0) {
            const int i = u / B, f = sel_kf(pk, i);
            const DevKf &K = pk.kf[f];
            const DevCand &c = wk.cand[u - i * B];
            S.new_tab = f != S.cur_f;
            S.cur_f = f;
            if (S.new_tab) {
                fence_proxy_async();
                mbar_expect_tx(&S.mbar, (uint32_t)K.tab_bytes);
                bulk_g2s(tab, pk.k1tab + K.tab_off, (uint32_t)K.tab_bytes, &S.mbar);
            }
            if (with_terms && pk.n_covis > 0 && K.n_kp > 0) {  // covisible pixels of this keyframe's keypoints: wanted in L2 ~50 us from now
                const unsigned long long a0 = (unsigned long long)(pk.covis_uv + K.kp_off * pk.n_covis);
                const unsigned long long a = a0 & ~15ull, e = (a0 + 8ull * K.n_kp * pk.n_covis) & ~15ull;
                if (e > a) bulk_prefetch_l2(reinterpret_cast<const void *>(a), (uint32_t)(e - a));
            }
            const double fx = K.fx, cx = K.cx, cy = K.cy;
            double ru[4], rv[4], rz[4];
            for (int j = 0; j < 3; ++j) {
                ru[j] = fx * c.R[j] + cx * c.R[6 + j];
                rv[j] = fx * c.R[3 + j] + cy * c.R[6 + j];
                rz[j] = c.R[6 + j];
            }
            ru[3] = fx * c.t[0] + cx * c.t[2];
            rv[3] = fx * c.t[1] + cy * c.t[2];
            rz[3] = c.t[2];
            for (int j = 0; j < 4; ++j) { S.mu[j] = (float)ru[j]; S.mv[j] = (float)rv[j]; S.mz[j] = (float)rz[j]; }
            // float32 error model of the fast path (DESIGN.md §K1): 3 FMAs + rounded matrix entries
            const double eps = 1.1920928955078125e-07, pm = K.pmax;
            const double Az = (fabs(rz[0]) + fabs(rz[1]) + fabs(rz[2])) * pm + fabs(rz[3]);
            const double Au = (fabs(ru[0]) + fabs(ru[1]) + fabs(ru[2])) * pm + fabs(ru[3]);
            const double Av = (fabs(rv[0]) + fabs(rv[1]) + fabs(rv[2])) * pm + fabs(rv[3]);
            const double ez = 4 * eps * Az, eu = 4 * eps * fmax(Au, Av);
            const double Umax = (double)max(K.W, K.H) + 8.0;
            const double zmin = (eu + Umax * ez) / ((double)kFastErrPx - Umax * 3 * eps);
            S.zmin = (float)(zmin * 1.0001) + 1e-30f;
            S.ez = (float)(ez * 1.0001);
            S.ub_u = (float)(((double)K.W + 2.0) * (zmin + ez) + eu);
            S.ub_v = (float)(((double)K.H + 2.0) * (zmin + ez) + eu);
            S.u_hi = (float)(kBmCell * (K.bm_wpr * 32 - 1));  // never index past the row
            S.u_hi = fminf(S.u_hi, (float)(K.W + kBmCell));
            S.v_hi = (float)(K.H + kBmCell);
            // Half-spaces every point that can pass the pre-cull satisfies (main case g_i >= 0; points of
            // the thin slab z <= zmin only satisfy g_i >= -m, so -m is the threshold).
            {
                const float uh = S.u_hi, vh = S.v_hi, two = (float)kBmCell;
                const float rzx = S.mz[0], rzy = S.mz[1], rzz = S.mz[2], rzw = S.mz[3];
                S.plane[0] = make_float4(rzx, rzy, rzz, rzw);
                S.plane[1] = make_float4(S.mu[0] + two * rzx, S.mu[1] + two * rzy, S.mu[2] + two * rzz, S.mu[3] + two * rzw);
                S.plane[2] = make_float4(uh * rzx - S.mu[0], uh * rzy - S.mu[1], uh * rzz - S.mu[2], uh * rzw - S.mu[3]);
                S.plane[3] = make_float4(S.mv[0] + two * rzx, S.mv[1] + two * rzy, S.mv[2] + two * rzz, S.mv[3] + two * rzw);
                S.plane[4] = make_float4(vh * rzx - S.mv[0], vh * rzy - S.mv[1], vh * rzz - S.mv[2], vh * rzw - S.mv[3]);
                const float mslab_u = S.ub_u + (uh + two) * (S.ez + S.zmin), mslab_v = S.ub_v + (vh + two) * (S.ez + S.zmin);
                S.thr[0] = -S.ez;
                S.thr[1] = -mslab_u; S.thr[2] = -mslab_u;
                S.thr[3] = -mslab_v; S.thr[4] = -mslab_v;
            }
            S.n_surv = 0; S.overflow = 0; S.n_groups = 0; S.n_match = 0; S.next_group = 0; S.he_val = 0.0; S.n_cells = 0;
            S.base_corr = 0; S.base_q = 0;
            S.covis_mask = K.covis_mask;
        }
    }
    for (int k = tid; k < max_kp; k += kThreads) { T.best_d2[k] = kInf64; T.best_key[k] = kNoKey; }
    __syncthreads();
    const int unit = S.unit;
    if (unit < 0) break;
    const int fi = unit / B, f = sel_kf(pk, fi), b = unit - fi * B;
    const DevKf K = pk.kf[f];
    const DevCand &c = wk.cand[b];
    const bool new_tab = S.new_tab != 0;
    float4 *const rec = wk.k1_rec + (size_t)blockIdx.x * kSurvCap;            // this CTA's survivor records
    ulonglong2 *const matches = wk.k1_match + (size_t)blockIdx.x * kMatchCap;  // ... and match list (both stay in L2)
    {
        const K1Tab tl = k1tab_layout(K.n_kp, K.bm_wpr * K.bm_rows, K.gw * K.gh);
        T.kp = reinterpret_cast<const float2 *>(tab);
        T.bm = reinterpret_cast<const uint32_t *>(tab + tl.off_bm);
        T.gstart = reinterpret_cast<const unsigned short *>(tab + tl.off_gs);
        T.gkp = reinterpret_cast<const unsigned short *>(tab + tl.off_gk);
        T.has_mp = reinterpret_cast<const uint32_t *>(tab + tl.off_mp);
    }
    long long clk[8];
    const bool timing = wk.k1_clk != nullptr && tid == 0;
    if (timing) clk[0] = clock64();

    // the ticket of the NEXT chunk is drawn now, by a thread of another warp, so that its round trip to L2 is off the
    // critical path of the next prologue (only when this unit ends the chunk in hand; a CTA stops at its first failing ticket)
    if (tid == 32 && unit + 1 >= S.u_end) { S.next_ticket = atomicAdd(wk.k1_ticket, 1); S.have_next = 1; }

    // ---- phase A1: which 128-point groups can hold a visible point?  Level-1 cells (1024 points) one per THREAD first,
    // then one warp per visible cell tests its 32 leaf boxes, one per lane: two dependent round trips to the boxes in all.
    {
        const float4 *nlo = pk.node_lo + K.node_off, *nhi = pk.node_hi + K.node_off;
        const int n_l1 = (K.n_pad + 1023) >> 10;
        for (int n0 = 0; n0 < n_l1; n0 += kThreads) {
            const int node = n0 + tid;
            const bool vis = node < n_l1 && box_visible(S, nlo[K.n0 + node], nhi[K.n0 + node]);
            const unsigned vm = __ballot_sync(0xffffffffu, vis);
            if (vm) {
                int base = 0;
                if (lane == 0) base = atomicAdd(&S.n_cells, __popc(vm));
                base = __shfl_sync(0xffffffffu, base, 0);
                if (vis) T.cells[base + __popc(vm & ((1u << lane) - 1))] = (unsigned short)node;
            }
        }
        __syncthreads();
        const int nc = S.n_cells;
        for (int ci = warp; ci < nc; ci += kThreads / 32) {
            const int node = T.cells[ci];
            const bool lv = box_visible(S, nlo[node * 32 + lane], nhi[node * 32 + lane]);
            const unsigned lmask = __ballot_sync(0xffffffffu, lv);
            // lane g < 8 owns group g of the cell (leaves 4g .. 4g+3)
            const bool need = lane < 8 && ((lmask >> (4 * lane)) & 0xfu) && (node * 8 + lane) * 128 < K.n_pad;
            const unsigned gm = __ballot_sync(0xffffffffu, need);
            if (gm) {
                int base = 0;
                if (lane == 0) base = atomicAdd(&S.n_groups, __popc(gm));
                base = __shfl_sync(0xffffffffu, base, 0);
                if (need) T.groups[base + __popc(gm & ((1u << lane) - 1))] = (unsigned short)(node * 8 + lane);
            }
        }
    }
    __syncthreads();
    if (new_tab) {  // the tables have landed (every thread observes the completion itself)
        mbar_wait(&S.mbar, tab_phase);
        tab_phase ^= 1u;
    }
    if (timing) clk[1] = clock64();

    // ---- phase A2: stream the visible groups (SoA float4 loads, 12 B/point), float32 pre-cull
    {
        const float mu0 = S.mu[0], mu1 = S.mu[1], mu2 = S.mu[2], mu3 = S.mu[3];
        const float mv0 = S.mv[0], mv1 = S.mv[1], mv2 = S.mv[2], mv3 = S.mv[3];
        const float mz0 = S.mz[0], mz1 = S.mz[1], mz2 = S.mz[2], mz3 = S.mz[3];
        const float zmin = S.zmin, u_hi = S.u_hi, v_hi = S.v_hi, lo = -(float)kBmCell;
        const int wpr = K.bm_wpr, cu_max = K.bm_wpr * 32 - 1, cv_max = K.bm_rows - 1;
        const float4 *X = reinterpret_cast<const float4 *>(pk.px + K.pt_off);
        const float4 *Y = reinterpret_cast<const float4 *>(pk.py + K.pt_off);
        const float4 *Z = reinterpret_cast<const float4 *>(pk.pz + K.pt_off);
        const int ng = S.n_groups;
        // the hand-eye term only needs the candidate: one lane of the last warp evaluates it while the
        // other warps stream (groups are handed out dynamically, so nobody waits for that warp)
        if (with_terms && K.he_valid && tid == kThreads - 32) S.he_val = hand_eye_term(pk, c, f);
        // software-pipelined: the loads of the next group are in flight while the current one is culled
        int w = 0;
        if (lane == 0) w = atomicAdd(&S.next_group, 1);
        w = __shfl_sync(0xffffffffu, w, 0);
        float4 x4 = make_float4(0.f, 0.f, 0.f, 0.f), y4 = x4, z4 = x4;
        int i = 0;
        if (w < ng) {
            i = (int)T.groups[w] * 32 + lane;  // float4 index
            x4 = ld_stream_f4(X + i); y4 = ld_stream_f4(Y + i); z4 = ld_stream_f4(Z + i);
        }
        while (w < ng) {
            int wn = 0;
            if (lane == 0) wn = atomicAdd(&S.next_group, 1);
            wn = __shfl_sync(0xffffffffu, wn, 0);
            float4 xn = x4, yn = y4, zn = z4;
            int in = 0;
            if (wn < ng) {
                in = (int)T.groups[wn] * 32 + lane;
                xn = ld_stream_f4(X + in); yn = ld_stream_f4(Y + in); zn = ld_stream_f4(Z + in);
            }
            const float xs[4] = {x4.x, x4.y, x4.z, x4.w}, ys[4] = {y4.x, y4.y, y4.z, y4.w}, zs[4] = {z4.x, z4.y, z4.z, z4.w};
            unsigned pm = 0;  // which of this lane's four points survive
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float zc = fmaf(mz0, xs[e], fmaf(mz1, ys[e], fmaf(mz2, zs[e], mz3)));
                const float uz = fmaf(mu0, xs[e], fmaf(mu1, ys[e], fmaf(mu2, zs[e], mu3)));
                const float vz = fmaf(mv0, xs[e], fmaf(mv1, ys[e], fmaf(mv2, zs[e], mv3)));
                bool pass = false;
                if (zc > zmin) {
                    // inside the apron-extended image?  (no division for the points that are not)
                    if (uz >= lo * zc && uz < u_hi * zc && vz >= lo * zc && vz < v_hi * zc) {
                        const float inv = __frcp_rn(zc);
                        const int cu = min(max((int)floorf(uz * inv * (1.0f / kBmCell)) + 1, 0), cu_max);
                        const int cv = min(max((int)floorf(vz * inv * (1.0f / kBmCell)) + 1, 0), cv_max);
                        pass = (T.bm[cv * wpr + (cu >> 5)] >> (cu & 31)) & 1u;
                    }
                } else if (zc > -S.ez) {
                    // thin slab in front of the camera plane where the float32 bound does not hold: exact path decides
                    pass = fabsf(uz) <= S.ub_u && fabsf(vz) <= S.ub_v;
                }
                pm |= (pass ? 1u : 0u) << e;
            }
            // one warp-aggregated append per group (a single shared-memory atomic instead of up to four
            // dependent ones per lane); a survivor is recorded WITH its coordinates (16 B, stays in L2), so the
            // exact pass never gathers from the scan
            if (__ballot_sync(0xffffffffu, pm != 0)) {
                const int cnt = __popc(pm);
                int inc = cnt;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int t = __shfl_up_sync(0xffffffffu, inc, o);
                    if (lane >= o) inc += t;
                }
                int base = 0;
                if (lane == 31) base = atomicAdd(&S.n_surv, inc);
                base = __shfl_sync(0xffffffffu, base, 31);
                int pos = base + inc - cnt;
#pragma unroll
                for (int e = 0; e < 4; ++e)
                    if ((pm >> e) & 1u) {
                        if (pos < kSurvCap) rec[pos] = make_float4(xs[e], ys[e], zs[e], __uint_as_float((uint32_t)(i * 4 + e)));
                        else S.overflow = 1;
                        ++pos;
                    }
            }
            w = wn; i = in; x4 = xn; y4 = yn; z4 = zn;
        }
    }
    __syncthreads();
    if (timing) clk[2] = clock64();

    // ---- phases B/C: exact fp64 re-evaluation of the survivors, (d2, original index) minimum per keypoint
    const bool ovf = S.overflow != 0;  // > kSurvCap survivors (never seen on real shapes): every point goes through the exact path
    const int ns = ovf ? K.n_pts : min(S.n_surv, kSurvCap);
    const float *gx = pk.px + K.pt_off, *gy = pk.py + K.pt_off, *gz = pk.pz + K.pt_off;
    // record s: from the CTA's list, or (overflow) straight from the scan; the load of the NEXT record is in flight while
    // the current one is evaluated
    auto load_rec = [&](int s) -> float4 { return ovf ? make_float4(gx[s], gy[s], gz[s], __uint_as_float((uint32_t)s)) : rec[s]; };
    {
        float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
        if (tid < ns) r = load_rec(tid);
        for (int s = tid; s < ns; s += kThreads) {
            float4 rn = r;
            if (s + kThreads < ns) rn = load_rec(s + kThreads);
            exact_point<1>(pk, K, c, pr, T, r.x, r.y, r.z, __float_as_uint(r.w), ovf ? 0u : (uint32_t)s, matches, &S.n_match);
            r = rn;
        }
        __syncthreads();
        if (timing) clk[3] = clock64();
        const int nm = S.n_match;
        if (nm <= kMatchCap) {  // the usual case: among the recorded matches, the ones at the minimum compete on the index
            // four matches per thread and round: the gathers of the original indices overlap
            for (int i0 = tid; i0 < nm; i0 += 4 * kThreads) {
                unsigned long long lowk[4];
                uint32_t og[4];
                bool hit[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int i = i0 + q * kThreads;
                    hit[q] = false;
                    if (i < nm) {
                        const ulonglong2 m = matches[i];
                        lowk[q] = m.y;
                        hit[q] = m.x == T.best_d2[(uint32_t)(m.y >> 32)];
                    }
                }
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    if (hit[q]) og[q] = pk.orig[K.pt_off + ((uint32_t)(lowk[q] & 0xffffffffu) >> 12)];
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    if (hit[q]) atomicMin(&T.best_key[(uint32_t)(lowk[q] >> 32)], ((unsigned long long)og[q] << 32) | (lowk[q] & 0xffffffffull));
            }
        } else {
            for (int s = tid; s < ns; s += kThreads) {
                const float4 r2 = load_rec(s);
                exact_point<2>(pk, K, c, pr, T, r2.x, r2.y, r2.z, __float_as_uint(r2.w), ovf ? 0u : (uint32_t)s, matches, &S.n_match);
            }
        }
    }
    __syncthreads();
    if (ovf && tid == 0 && wk.overflow) atomicAdd(wk.overflow, 1);
    if (timing) clk[4] = clock64();

    // ---- phase D: corrset in keypoint order, query list = correspondences with a map point, and the 3-D/2-D term of
    // every correspondence (iba_global.cpp:291-328).  One block scan: thread t owns the consecutive keypoints
    // [t*per, (t+1)*per); nothing here gathers from HBM (keys and map-point flags in shared memory, point
    // coordinates from the CTA's records, covisible pixels prefetched into L2 by the prologue); the (correspondence,
    // covisible keyframe) pairs are dealt evenly to the threads.
    const unsigned long long *best_key = T.best_key;
    const long long out_base = (long long)b * pk.n_kp_total + K.kp_off;
    double s2d = 0, v2d = 0, c2d = 0;
    int ncorr = 0, nq = 0;
    bool kept = false;
    {
        const int per = (K.n_kp + kThreads - 1) / kThreads;
        const int k_lo = min(tid * per, K.n_kp), k_hi = min(k_lo + per, K.n_kp);
        int cc = 0, cq = 0;
        for (int k = k_lo; k < k_hi; ++k) {
            const bool has = best_key[k] != kNoKey;
            cc += has;
            cq += has && ((T.has_mp[k >> 5] >> (k & 31)) & 1u);
        }
        int ic = cc, iq = cq;  // inclusive warp scans
        for (int o = 1; o < 32; o <<= 1) {
            const int a = __shfl_up_sync(0xffffffffu, ic, o), a2 = __shfl_up_sync(0xffffffffu, iq, o);
            if (lane >= o) { ic += a; iq += a2; }
        }
        if (lane == 31) { S.warp_cnt[warp] = ic; S.warp_q[warp] = iq; }
        __syncthreads();
        int pc = ic - cc, pq = iq - cq, tc = 0, tq = 0;
        for (int w = 0; w < kThreads / 32; ++w) {
            if (w < warp) { pc += S.warp_cnt[w]; pq += S.warp_q[w]; }
            tc += S.warp_cnt[w]; tq += S.warp_q[w];
        }
        ncorr = tc; nq = tq;
        kept = ncorr >= pr.num_min_corr;  // iba_global.cpp:203
        const bool terms = kept && with_terms && pk.n_covis > 0;
        // (keypoint, position, slot) of correspondence i, for the pair loop below; the per-keypoint minima are dead by now
        unsigned long long *clist = T.best_d2;  // (last read in the tie pass, two barriers ago)
        for (int k = k_lo; k < k_hi; ++k) {
            const unsigned long long key = best_key[k];
            if (key == kNoKey) continue;
            const uint32_t low = (uint32_t)(key & 0xffffffffu), sp = low >> 12;
            wk.corr_kp[out_base + pc] = (uint32_t)k;
            wk.corr_pt[out_base + pc] = (uint32_t)(key >> 32);
            wk.corr_sp[out_base + pc] = sp;
            clist[pc] = ((unsigned long long)k << 32) | low;
            if ((T.has_mp[k >> 5] >> (k & 31)) & 1u) {
                wk.q_corr[out_base + pq] = (uint32_t)pc;
                wk.q_kpsp[out_base + pq] = make_uint2((uint32_t)k, sp);
                ++pq;
            }
            ++pc;
        }
        if (terms) {
            // 3-D/2-D term over (covisible keyframe) x (correspondence), the pairs dealt evenly to the threads
            __syncthreads();
            const int C = pk.n_covis;
            const unsigned cmask = S.covis_mask;
            const double fx = K.fx, fy = K.fy, cx = K.cx, cy = K.cy, W = K.W, H = K.H;
            for (int j = 0; j < C; ++j) {
                if (!((cmask >> j) & 1u)) continue;
                const float *rp = pk.relpose + ((long long)f * C + j) * 12;
                const float2 *uvj = pk.covis_uv + K.kp_off * C + j;
                for (int i = tid; i < ncorr; i += kThreads) {
                    const unsigned long long e = clist[i];
                    const uint32_t k = (uint32_t)(e >> 32), low = (uint32_t)(e & 0xffffffffu);
                    const float2 uv = uvj[(long long)k * C];
                    if (isnan(uv.x)) continue;
                    const float4 r = ovf ? make_float4(gx[low >> 12], gy[low >> 12], gz[low >> 12], 0.f) : rec[low & 0xfffu];
                    double p0x, p0y, p0z;
                    xform(c.R, c.t, (double)r.x, (double)r.y, (double)r.z, p0x, p0y, p0z);
                    const double p1x = dadd(dot3e((double)rp[0], (double)rp[1], (double)rp[2], p0x, p0y, p0z), dmul((double)rp[3], c.s));
                    const double p1y = dadd(dot3e((double)rp[4], (double)rp[5], (double)rp[6], p0x, p0y, p0z), dmul((double)rp[7], c.s));
                    const double p1z = dadd(dot3e((double)rp[8], (double)rp[9], (double)rp[10], p0x, p0y, p0z), dmul((double)rp[11], c.s));
                    const double ou = dadd(ddiv(dmul(fx, p1x), p1z), cx);
                    const double ov = dadd(ddiv(dmul(fy, p1y), p1z), cy);
                    if (!(ou >= 0 && ou < W && ov >= 0 && ov < H)) continue;
                    const double du = dsub(ou, (double)uv.x), dv = dsub(ov, (double)uv.y);
                    const double dist = sqrt(dadd(dmul(du, du), dmul(dv, dv)));
                    if (dist < pr.thr2d) { s2d += dist; v2d += 1.0; }
                    c2d += 1.0;
                }
            }
        }
    }
    if (timing) clk[5] = clock64();
    // fixed-order block reduction (deterministic)
    for (int o = 16; o; o >>= 1) {
        s2d += __shfl_down_sync(0xffffffffu, s2d, o);
        v2d += __shfl_down_sync(0xffffffffu, v2d, o);
        c2d += __shfl_down_sync(0xffffffffu, c2d, o);
    }
    if (lane == 0) { S.red[0][warp] = s2d; S.red[1][warp] = v2d; S.red[2][warp] = c2d; }
    __syncthreads();
    if (timing) clk[6] = clock64();
    if (tid == 0) {
        FrameRec r;
        r.s2d = r.v2d = r.c2d = 0;
        for (int w = 0; w < kThreads / 32; ++w) { r.s2d += S.red[0][w]; r.v2d += S.red[1][w]; r.c2d += S.red[2][w]; }
        r.she = 0; r.che = 0;
        if (kept && K.he_valid && with_terms) { r.she = S.he_val; r.che = 1; }
        r.kept = kept ? 1.0 : 0.0;
        r.ncorr = kept ? (double)ncorr : 0.0;
        r.nq = kept ? (double)nq : 0.0;
        wk.frame[(long long)b * pk.n_kf + f] = r;
        wk.n_corr[(long long)b * pk.n_kf + f] = ncorr;
        wk.n_q[(long long)b * pk.n_kf + f] = kept ? nq : 0;
        if (timing) {
            long long *o = wk.k1_clk + (long long)unit * 8;
            for (int i = 0; i < 6; ++i) o[i] = clk[i + 1] - clk[i];
            o[6] = clock64() - clk[6];
            o[7] = clk[0] - clk_top;  // thread 0's prologue (ticket, fast rows, bulk copy issued) incl. the barrier behind it
        }
    }
    }  // persistent loop
}

}  // namespace

size_t assoc2d_smem_bytes(int max_kp, int max_tab_bytes, int max_groups) {
    return ((sizeof(Smem) + 15) & ~size_t(15)) + (size_t)max_tab_bytes + (size_t)max_kp * 16 + 2 * (size_t)max_groups + 2 * (size_t)(max_groups / 8 + 1) + 16;
}

// The opt-in dynamic shared-memory limit is a per-function, per-device attribute shared by every
// context of the process: only ever raise it.
cudaError_t assoc2d_configure(size_t smem) {
    static size_t granted[64] = {0};
    static std::mutex mu;  // contexts of different devices / threads share this table
    std::lock_guard<std::mutex> lk(mu);
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
    if (smem <= granted[dev]) return cudaSuccess;
    e = cudaFuncSetAttribute(k_assoc2d, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) granted[dev] = smem;
    return e;
}

cudaError_t launch_assoc2d(const DevPack &pk, const DevWork &wk, const DevParams &pr, int B, size_t smem, int max_kp, int max_tab_bytes,
                           int max_groups, cudaStream_t st, int with_terms) {
    if (B <= 0 || pk.n_sel <= 0) return cudaSuccess;
    const long long n_units = (long long)pk.n_sel * B;  // unit = selection position * B + candidate
    if (n_units > 0x7fffffffll || wk.k1_slots <= 0) return cudaErrorInvalidValue;
    // candidates of one keyframe are consecutive units: a chunk keeps the keyframe's tables in shared memory
    const int chunk = B >= 64 ? 8 : (B >= 16 ? 4 : (B >= 4 ? 2 : 1));
    const long long n_chunks = (n_units + chunk - 1) / chunk;
    const unsigned grid = (unsigned)std::min<long long>(n_chunks, wk.k1_slots);
    k_assoc2d<<<grid, kThreads, smem, st>>>(pk, wk, pr, B, with_terms, (int)n_units, chunk, max_kp, max_tab_bytes, max_groups);
    return cudaGetLastError();
}

}  // namespace stl
