// assoc2d_split.cu — K1 as three kernels, for the keyframes whose K1 tables do not fit the one-kernel K1's shared memory
// (stl_allow_oversize_keyframes; STL_K1_OVERSIZE=all or STL_K1_SPLIT=1 route every keyframe here).  Nothing it keeps in
// shared memory grows with the image: the stream holds one BAND of the keypoint bitmap (kK1BandWords), and the exact and
// correspondence passes keep their per-keypoint tables in global memory.
// Status: bit-identical results to the one-kernel form (assoc2d.cu), but 13 % SLOWER than it at the KITTI-00 shape when
// routed there — k_stream 0.152 ms (instruction-bound, 80 % issue), k_exact 0.213 ms and k_corr 0.137 ms (both bound by
// chains of dependent L2 / DRAM round trips at 23 % issue), against 0.447 ms in one kernel (profiles/r02_negative_results.txt).
//
// Same result as k_assoc2d (assoc2d.cu), i.e. per (candidate, keyframe):
//   TransformPointCloud + FindProjectCorrespondences   include/pointcloud.h:82-86, src/examples/iba_global.cpp:55-96
//   frame gate, hand-eye term, covisible term           src/examples/iba_global.cpp:203,264-276,291-328
// but every phase runs on the grid shape that suits it:
//   K1a k_stream   bands x S CTAs per unit stream the scan (SoA float4 loads, 12 B/point) through the float32 pre-cull and
//                  the keypoint bitmap.  A CTA holds one band of bitmap rows, culls the KD cells with the v-range of its
//                  band, and tests a point's bit only when the point's cell row falls in its band (the bitmap is dilated
//                  by max_pixel_dist + 0.25 px, so every point is decided in exactly one band; the z < zmin slab goes to
//                  the exact pass from band 0).  Band + group list + a local survivor list stay under ~49 KB of shared
//                  memory, so four CTAs fit an SM.  Survivors (1-2 % of the points) go to a per-unit list in global memory.
//   K1b k_exact    one THREAD per survivor: the reference's exact fp64 projection, the keypoints of the 8 px grid cells
//                  around it, atomicMin of the squared distance per keypoint on a table in global memory (L2 atomics),
//                  every match appended to the unit's match list.
//   K1c k_corr     one CTA per unit: ties among the matches resolved by (original index, position), corrset compacted in
//                  keypoint order, query list, covisible term over (correspondence, covisible keyframe) pairs, hand-eye
//                  term, per-unit record.
// With one candidate over 1500 keyframes the one-kernel form spends 36 % of a CTA's life streaming and the rest in
// latency-bound phases of a few thousand items, at 2 CTAs/SM and 5.07 waves (profiles/r02_negative_results.txt); split,
// the stream is bound by HBM and the item-parallel phases by their instruction count.
#include <cstdlib>
#include <mutex>

#include "../../include/stlcalib.h"
#include "kernels.h"
#include "se3.cuh"

namespace stl {
namespace {

constexpr int kStreamThreads = 256;
constexpr int kExactThreads = 256;
constexpr int kCorrThreads = 256;
// the 3-D/2-D term is summed in the order of the one-kernel K1 (assoc2d.cu, CTAs of 512 threads), each k_corr thread playing
// two of its threads, so that STL_K1_SPLIT=1 changes no bit of the record
constexpr int kTermLanes = 512;
static_assert(kTermLanes == 2 * kCorrThreads, "k_corr plays two threads of the one-kernel K1 each");
constexpr int kLocalSurv = kK1SurvCap;  // survivors a stream CTA holds in shared memory (flushed once, at its end; beyond: straight to the unit's list)
constexpr unsigned long long kNoKey = 0xffffffffffffffffull;

struct Fast {  // float32 projection rows, error bounds and the culling half-spaces of one (candidate, keyframe)
    float mu[4], mv[4], mz[4];
    float zmin, ub_u, ub_v, ez, u_hi, v_hi;
    float4 plane[5];
    float thr[5];
};

// The float32 error model of the pre-cull (DESIGN.md K1): identical to the prologue of k_assoc2d.
__device__ void make_fast(const DevKf &K, const DevCand &c, Fast &S) {
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
    S.u_hi = (float)(kBmCell * (K.bm_wpr * 32 - 1));
    S.u_hi = fminf(S.u_hi, (float)(K.W + kBmCell));
    S.v_hi = (float)(K.H + kBmCell);
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

__device__ __forceinline__ bool box_visible(const Fast &S, float4 lo, float4 hi) {
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

// per-unit counters in global memory
struct UnitCnt { int n_surv, n_match, overflow, pad; };

// ------------------------------------------------------------------------------------------------ K1a
struct StreamSmem {
    Fast F;
    int n_groups, next_group, n_local, flush_base;
};

// The cull of band [r0, r1) of bitmap rows: cell row cv = floor(v / kBmCell) + 1 covers v in [kBmCell (cv - 1), kBmCell cv), so
// the band's points have v in [kBmCell (r0 - 1), kBmCell (r1 - 1)); the v half-spaces are moved to that range widened by one
// cell on either side, the margin the image range itself has (-kBmCell, H + kBmCell).  The first and last band keep the
// image's own bounds; the thresholds stay those of the slab z <= zmin (conservative for every band, exact for band 0).
__device__ void narrow_to_band(Fast &S, int r0, int r1, int rows) {
    const float rzx = S.mz[0], rzy = S.mz[1], rzz = S.mz[2], rzw = S.mz[3];
    if (r0 > 0) {
        const float vl = (float)(kBmCell * (r0 - 2));
        S.plane[3] = make_float4(S.mv[0] - vl * rzx, S.mv[1] - vl * rzy, S.mv[2] - vl * rzz, S.mv[3] - vl * rzw);
    }
    if (r1 < rows) {
        const float vh = fminf((float)(kBmCell * r1), S.v_hi);
        S.plane[4] = make_float4(vh * rzx - S.mv[0], vh * rzy - S.mv[1], vh * rzz - S.mv[2], vh * rzw - S.mv[3]);
    }
}

// grid: ((unit * max_bands + band) * S + sub), unit = oversize selection position * B + candidate; CTAs of bands the
// keyframe does not have leave at once
__global__ void __launch_bounds__(kStreamThreads, 6)
k_stream(const DevPack pk, const DevWork wk, const int B, const int S_sub, const int max_bands) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int sub = blockIdx.x % S_sub, ub = blockIdx.x / S_sub, band = ub % max_bands, unit = ub / max_bands;
    const int oi = unit / B, b = unit - oi * B, o = pk.ov_sel[oi];
    const OvKf O = pk.ov[o];
    if (band >= O.n_bands) return;
    const DevKf K = pk.kf[O.f];
    const DevCand &c = wk.cand[b];
    const int wpr = K.bm_wpr, band_rows = k1_band_rows(wpr), r0 = band * band_rows, r1 = min(r0 + band_rows, K.bm_rows);
    StreamSmem &S = *reinterpret_cast<StreamSmem *>(smem_raw);
    unsigned char *p = smem_raw + ((sizeof(StreamSmem) + 15) & ~size_t(15));
    // the band's words, then the lists: at most min(band_rows, bm_rows) rows, as assoc2d_split_smem_bytes is given
    uint32_t *bm = reinterpret_cast<uint32_t *>(p); p += 4 * (size_t)wpr * min(band_rows, K.bm_rows);
    uint32_t *surv = reinterpret_cast<uint32_t *>(p); p += 4 * (size_t)kLocalSurv;
    unsigned short *groups = reinterpret_cast<unsigned short *>(p);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    UnitCnt *cnt = reinterpret_cast<UnitCnt *>(wk.k1_cnt) + (long long)b * pk.n_ov + o;
    uint32_t *gsurv = wk.k1_surv + (long long)b * pk.n_ov_surv + O.surv_off;
    const int surv_cap = O.surv_cap;

    if (tid == 0) {
        make_fast(K, c, S.F);
        narrow_to_band(S.F, r0, r1, K.bm_rows);
        S.n_groups = 0; S.next_group = 0; S.n_local = 0; S.flush_base = 0;
    }
    {
        const uint32_t *bmg = pk.bitmap + K.bm_off + (long long)r0 * wpr;
        const int nw = (r1 - r0) * wpr;
        for (int i = tid; i < nw; i += kStreamThreads) bm[i] = bmg[i];
    }
    __syncthreads();

    // which 128-point groups of this CTA's share can hold a visible point?  One warp per level-1 cell (1024 points)
    {
        const float4 *nlo = pk.node_lo + K.node_off, *nhi = pk.node_hi + K.node_off;
        const int n_l1 = (K.n_pad + 1023) >> 10;
        for (int node = sub + S_sub * warp; node < n_l1; node += S_sub * (kStreamThreads / 32)) {
            if (!box_visible(S.F, nlo[K.n0 + node], nhi[K.n0 + node])) continue;
            const bool lv = box_visible(S.F, nlo[node * 32 + lane], nhi[node * 32 + lane]);
            const unsigned lmask = __ballot_sync(0xffffffffu, lv);
            const bool need = lane < 8 && ((lmask >> (4 * lane)) & 0xfu) && (node * 8 + lane) * 128 < K.n_pad;
            const unsigned gm = __ballot_sync(0xffffffffu, need);
            if (gm) {
                int base = 0;
                if (lane == 0) base = atomicAdd(&S.n_groups, __popc(gm));
                base = __shfl_sync(0xffffffffu, base, 0);
                if (need) groups[base + __popc(gm & ((1u << lane) - 1))] = (unsigned short)(node * 8 + lane);
            }
        }
    }
    __syncthreads();

    {
        const Fast &F = S.F;
        const float mu0 = F.mu[0], mu1 = F.mu[1], mu2 = F.mu[2], mu3 = F.mu[3];
        const float mv0 = F.mv[0], mv1 = F.mv[1], mv2 = F.mv[2], mv3 = F.mv[3];
        const float mz0 = F.mz[0], mz1 = F.mz[1], mz2 = F.mz[2], mz3 = F.mz[3];
        const float zmin = F.zmin, u_hi = F.u_hi, v_hi = F.v_hi, lo = -(float)kBmCell, ezs = F.ez, ubu = F.ub_u, ubv = F.ub_v;
        const int cu_max = wpr * 32 - 1, cv_max = K.bm_rows - 1;
        const bool slab = band == 0;  // the z < zmin slab is passed to the exact pass by the first band only
        const float4 *X = reinterpret_cast<const float4 *>(pk.px + K.pt_off);
        const float4 *Y = reinterpret_cast<const float4 *>(pk.py + K.pt_off);
        const float4 *Z = reinterpret_cast<const float4 *>(pk.pz + K.pt_off);
        const int ng = S.n_groups;
        int w = 0;
        if (lane == 0) w = atomicAdd(&S.next_group, 1);
        w = __shfl_sync(0xffffffffu, w, 0);
        float4 x4 = make_float4(0.f, 0.f, 0.f, 0.f), y4 = x4, z4 = x4;
        int i = 0;
        if (w < ng) {
            i = (int)groups[w] * 32 + lane;
            x4 = ld_stream_f4(X + i); y4 = ld_stream_f4(Y + i); z4 = ld_stream_f4(Z + i);
        }
        while (w < ng) {  // software-pipelined: the next group's loads are in flight while this one is culled
            int wn = 0;
            if (lane == 0) wn = atomicAdd(&S.next_group, 1);
            wn = __shfl_sync(0xffffffffu, wn, 0);
            float4 xn = x4, yn = y4, zn = z4;
            int in = 0;
            if (wn < ng) {
                in = (int)groups[wn] * 32 + lane;
                xn = ld_stream_f4(X + in); yn = ld_stream_f4(Y + in); zn = ld_stream_f4(Z + in);
            }
            const float xs[4] = {x4.x, x4.y, x4.z, x4.w}, ys[4] = {y4.x, y4.y, y4.z, y4.w}, zs[4] = {z4.x, z4.y, z4.z, z4.w};
            unsigned pm = 0;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float zc = fmaf(mz0, xs[e], fmaf(mz1, ys[e], fmaf(mz2, zs[e], mz3)));
                const float uz = fmaf(mu0, xs[e], fmaf(mu1, ys[e], fmaf(mu2, zs[e], mu3)));
                const float vz = fmaf(mv0, xs[e], fmaf(mv1, ys[e], fmaf(mv2, zs[e], mv3)));
                bool pass = false;
                if (zc > zmin) {
                    if (uz >= lo * zc && uz < u_hi * zc && vz >= lo * zc && vz < v_hi * zc) {
                        const float inv = __frcp_rn(zc);
                        const int cu = min(max((int)floorf(uz * inv * (1.0f / kBmCell)) + 1, 0), cu_max);
                        const int cv = min(max((int)floorf(vz * inv * (1.0f / kBmCell)) + 1, 0), cv_max);
                        pass = cv >= r0 && cv < r1 && ((bm[(cv - r0) * wpr + (cu >> 5)] >> (cu & 31)) & 1u);
                    }
                } else if (slab && zc > -ezs) {
                    pass = fabsf(uz) <= ubu && fabsf(vz) <= ubv;
                }
                pm |= (pass ? 1u : 0u) << e;
            }
            if (__ballot_sync(0xffffffffu, pm != 0)) {
                const int cntl = __popc(pm);
                int inc = cntl;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int t = __shfl_up_sync(0xffffffffu, inc, o);
                    if (lane >= o) inc += t;
                }
                int base = 0;
                if (lane == 31) base = atomicAdd(&S.n_local, inc);
                base = __shfl_sync(0xffffffffu, base, 31);
                int pos = base + inc - cntl;
#pragma unroll
                for (int e = 0; e < 4; ++e)
                    if ((pm >> e) & 1u) {
                        if (pos < kLocalSurv) {
                            surv[pos] = (uint32_t)(i * 4 + e);
                        } else {  // the CTA's list is full: straight to the unit's list
                            const int g = atomicAdd(&cnt->n_surv, 1);
                            if (g < surv_cap) gsurv[g] = (uint32_t)(i * 4 + e);
                            else atomicExch(&cnt->overflow, 1);
                        }
                        ++pos;
                    }
            }
            w = wn; i = in; x4 = xn; y4 = yn; z4 = zn;
        }
    }
    __syncthreads();
    // flush: one reservation in the unit's global list per CTA
    const int nl = min(S.n_local, kLocalSurv);
    if (tid == 0) {
        const int base = atomicAdd(&cnt->n_surv, nl);
        S.flush_base = base;
        if (base + nl > surv_cap) atomicExch(&cnt->overflow, 1);
    }
    __syncthreads();
    const int fb = S.flush_base;
    for (int s = tid; s < nl; s += kStreamThreads)
        if (fb + s < surv_cap) gsurv[fb + s] = surv[s];
}

// ------------------------------------------------------------------------------------------------ K1b
template <bool STABLE>
__device__ __forceinline__ bool exact_project(const DevCand &c, double fx, double cx, double cy, double W, double H, float xf, float yf,
                                              float zf, double &u, double &v) {
    double xc, yc, zc;
    xform(c.R, c.t, (double)xf, (double)yf, (double)zf, xc, yc, zc);
    if (!(zc > 0.0)) return false;
    u = ddiv(dadd(dmul(fx, xc), dmul(cx, zc)), zc);
    v = ddiv(dadd(dmul(fx, yc), dmul(cy, zc)), zc);  // fx, not fy (iba_global.cpp:73)
    if (STABLE) {  // iba_global_stable.cpp:92-94
        const double ru = round(u), rv = round(v);
        return (0.0 <= ru && ru < W && 0.0 <= rv && rv < H);
    }
    return (0.0 <= u && u < W && 0.0 <= v && v < H);
}

// PASS 1: atomicMin of the squared distance per keypoint + match list; PASS 2 (match list overflowed): ties by recomputation
template <int PASS>
__device__ __forceinline__ void exact_point(const DevPack &pk, const DevKf &K, const DevCand &c, const DevParams &pr, unsigned long long *best_d2,
                                            unsigned long long *best_key, uint32_t si, ulonglong2 *__restrict__ matches, int *n_match, int match_cap) {
    const long long g = K.pt_off + si;
    const float xf = pk.px[g], yf = pk.py[g], zf = pk.pz[g];
    double u, v;
    const bool stable = pk.kp_xyd != nullptr;
    if (stable ? !exact_project<true>(c, (double)K.fx, (double)K.cx, (double)K.cy, (double)K.W, (double)K.H, xf, yf, zf, u, v)
               : !exact_project<false>(c, (double)K.fx, (double)K.cx, (double)K.cy, (double)K.W, (double)K.H, xf, yf, zf, u, v)) return;
    const uint32_t *gstart = pk.grid_start + K.grid_off, *gkp = pk.grid_kp + K.kp_off;
    const double rp = sqrt(pr.max_pixel_dist2) + (stable ? 1e-3 : 1e-6);
    int gx0 = (int)floor((u - rp) * (1.0 / kGridCell)), gx1 = (int)floor((u + rp) * (1.0 / kGridCell));
    int gy0 = (int)floor((v - rp) * (1.0 / kGridCell)), gy1 = (int)floor((v + rp) * (1.0 / kGridCell));
    gx0 = max(gx0, 0); gy0 = max(gy0, 0); gx1 = min(gx1, K.gw - 1); gy1 = min(gy1, K.gh - 1);
    for (int gy = gy0; gy <= gy1; ++gy) {
        const int a = (int)gstart[gy * K.gw + gx0], b = (int)gstart[gy * K.gw + gx1 + 1];  // cells of one row are contiguous
        for (int j = a; j < b; ++j) {
            const int k = (int)gkp[j];
            double qx, qy;
            if (stable) { const double2 q = pk.kp_xyd[K.kp_off + k]; qx = q.x; qy = q.y; }
            else { const float2 q = pk.kp_xy[K.kp_off + k]; qx = (double)q.x; qy = (double)q.y; }
            const double dx = dsub(qx, u), dy = dsub(qy, v);
            const double d2 = dadd(dmul(dx, dx), dmul(dy, dy));  // nanoflann.hpp:524-535, query - data
            if (d2 <= pr.max_pixel_dist2) {
                const unsigned long long bits = (unsigned long long)__double_as_longlong(d2);
                if (PASS == 1) {
                    atomicMin(&best_d2[k], bits);
                    const int slot = atomicAdd(n_match, 1);
                    if (slot < match_cap) matches[slot] = make_ulonglong2(bits, ((unsigned long long)k << 32) | si);
                } else if (bits == __ldcg(&best_d2[k])) {
                    atomicMin(&best_key[k], ((unsigned long long)pk.orig[g] << 32) | si);
                }
            }
        }
    }
}

// grid: (units, chunks per unit): thread per survivor
__global__ void __launch_bounds__(kExactThreads)
k_exact(const DevPack pk, const DevWork wk, const DevParams pr, const int B) {
    const int unit = blockIdx.x;
    const int oi = unit / B, b = unit - oi * B, o = pk.ov_sel[oi];
    const OvKf O = pk.ov[o];
    UnitCnt *cnt = reinterpret_cast<UnitCnt *>(wk.k1_cnt) + (long long)b * pk.n_ov + o;
    const DevKf K = pk.kf[O.f];
    const bool ovf = cnt->overflow != 0;
    const int ns = ovf ? K.n_pts : min(cnt->n_surv, O.surv_cap);
    const int first = blockIdx.y * kExactThreads + threadIdx.x;
    if (first >= ns) return;
    const DevCand &c = wk.cand[b];
    const uint32_t *gsurv = wk.k1_surv + (long long)b * pk.n_ov_surv + O.surv_off;
    unsigned long long *best_d2 = wk.k1_best_d2 + (long long)b * pk.n_ov_kp + O.kp_off;
    ulonglong2 *matches = wk.k1_ov_match + (long long)b * pk.n_ov_match + O.match_off;
    for (int s = first; s < ns; s += gridDim.y * kExactThreads)
        exact_point<1>(pk, K, c, pr, best_d2, nullptr, ovf ? (uint32_t)s : gsurv[s], matches, &cnt->n_match, O.match_cap);
}

// ------------------------------------------------------------------------------------------------ K1c
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

struct CorrSmem {
    int warp_cnt[kCorrThreads / 32], warp_q[kCorrThreads / 32];
    int ncorr, nq;
    double he_val;
    double red[3][kTermLanes / 32];
    float rel[STL_MAX_COVIS][12];
    int cval[STL_MAX_COVIS];
};

// grid: units
__global__ void __launch_bounds__(kCorrThreads)
k_corr(const DevPack pk, const DevWork wk, const DevParams pr, const int B, const int with_terms) {
    __shared__ CorrSmem S;
    const int unit = blockIdx.x;
    const int oi = unit / B, b = unit - oi * B, o = pk.ov_sel[oi];
    const OvKf O = pk.ov[o];
    const int f = O.f;
    const long long urec = (long long)b * pk.n_kf + f;  // the records every K1 writes
    UnitCnt *cnt = reinterpret_cast<UnitCnt *>(wk.k1_cnt) + (long long)b * pk.n_ov + o;
    const DevKf K = pk.kf[f];
    const DevCand &c = wk.cand[b];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    unsigned long long *best_d2 = wk.k1_best_d2 + (long long)b * pk.n_ov_kp + O.kp_off;
    unsigned long long *best_key = wk.k1_best_key + (long long)b * pk.n_ov_kp + O.kp_off;
    const ulonglong2 *matches = wk.k1_ov_match + (long long)b * pk.n_ov_match + O.match_off;
    const int C = pk.n_covis;
    if (tid >= 32 && tid < 32 + C) {
        const int j = tid - 32;
        S.cval[j] = pk.covis_valid[f * C + j];
        const float *rp = pk.relpose + ((long long)f * C + j) * 12;
        for (int t = 0; t < 12; ++t) S.rel[j][t] = rp[t];
    }
    // the hand-eye term only needs the candidate: one thread evaluates it while the others resolve the ties
    if (tid == kCorrThreads - 1) S.he_val = (with_terms && K.he_valid) ? hand_eye_term(pk, c, f) : 0.0;

    // ---- ties: among the recorded matches, the ones at the minimum compete on (original index, position)
    const int nm = cnt->n_match;
    if (nm <= O.match_cap) {
        for (int i = tid; i < nm; i += kCorrThreads) {
            const ulonglong2 m = matches[i];
            const uint32_t k = (uint32_t)(m.y >> 32), si = (uint32_t)(m.y & 0xffffffffu);
            if (m.x == __ldcg(&best_d2[k])) atomicMin(&best_key[k], ((unsigned long long)pk.orig[K.pt_off + si] << 32) | si);
        }
    } else {  // match list overflowed: recompute
        const bool ovf = cnt->overflow != 0;
        const int ns = ovf ? K.n_pts : min(cnt->n_surv, O.surv_cap);
        const uint32_t *gsurv = wk.k1_surv + (long long)b * pk.n_ov_surv + O.surv_off;
        for (int s = tid; s < ns; s += kCorrThreads)
            exact_point<2>(pk, K, c, pr, best_d2, best_key, ovf ? (uint32_t)s : gsurv[s], nullptr, nullptr, 0);
    }
    __threadfence_block();
    __syncthreads();
    if (tid == 0 && cnt->overflow && wk.overflow) atomicAdd(wk.overflow, 1);

    // ---- corrset in keypoint order, query list = correspondences with a map point (one block scan)
    const long long out_base = (long long)b * pk.n_kp_total + K.kp_off;
    const float *mp = pk.kp_mp + K.kp_off * 3;
    {
        const int per = (K.n_kp + kCorrThreads - 1) / kCorrThreads;
        const int k_lo = min(tid * per, K.n_kp), k_hi = min(k_lo + per, K.n_kp);
        int cc = 0, cq = 0;
        for (int k = k_lo; k < k_hi; ++k) {
            const bool has = __ldcg(&best_key[k]) != kNoKey;
            cc += has;
            cq += has && !isnan(mp[k * 3]);
        }
        int ic = cc, iq = cq;
        for (int o = 1; o < 32; o <<= 1) {
            const int a = __shfl_up_sync(0xffffffffu, ic, o), a2 = __shfl_up_sync(0xffffffffu, iq, o);
            if (lane >= o) { ic += a; iq += a2; }
        }
        if (lane == 31) { S.warp_cnt[warp] = ic; S.warp_q[warp] = iq; }
        __syncthreads();
        int pc = ic - cc, pq = iq - cq, tc = 0, tq = 0;
        for (int w = 0; w < kCorrThreads / 32; ++w) {
            if (w < warp) { pc += S.warp_cnt[w]; pq += S.warp_q[w]; }
            tc += S.warp_cnt[w]; tq += S.warp_q[w];
        }
        for (int k = k_lo; k < k_hi; ++k) {
            const unsigned long long key = __ldcg(&best_key[k]);
            if (key == kNoKey) continue;
            wk.corr_kp[out_base + pc] = (uint32_t)k;
            wk.corr_pt[out_base + pc] = (uint32_t)(key >> 32);
            wk.corr_sp[out_base + pc] = (uint32_t)(key & 0xffffffffu);
            if (!isnan(mp[k * 3])) {
                wk.q_corr[out_base + pq] = (uint32_t)pc;
                wk.q_kpsp[out_base + pq] = make_uint2((uint32_t)k, (uint32_t)(key & 0xffffffffu));
                ++pq;
            }
            ++pc;
        }
        if (tid == 0) { S.ncorr = tc; S.nq = tq; }
        __syncthreads();  // also publishes the lists to the covisible phase below
    }
    const int ncorr = S.ncorr, nq = S.nq;
    const bool kept = ncorr >= pr.num_min_corr;  // iba_global.cpp:203

    // ---- 3-D/2-D term over (correspondence, covisible keyframe) pairs, iba_global.cpp:291-328, in the one-kernel K1's order:
    // covisible keyframe j outer, correspondence i = v, v + 512, ... inner for its thread v; here thread t plays v = t (h = 0)
    // and v = t + 256 (h = 1), and the reduction below is that kernel's tree over its 16 warps
    double s2d[2] = {0, 0}, v2d[2] = {0, 0}, c2d[2] = {0, 0};
    if (kept && with_terms && C > 0) {
        const double fx = K.fx, fy = K.fy, cx = K.cx, cy = K.cy, W = K.W, H = K.H;
        for (int j = 0; j < C; ++j) {
            if (!S.cval[j]) continue;
            const float *rp = S.rel[j];
            for (int h = 0; h < 2; ++h) {
                for (int i = tid + h * kCorrThreads; i < ncorr; i += kTermLanes) {
                    const int k = (int)wk.corr_kp[out_base + i];
                    const float2 uv = pk.covis_uv[(K.kp_off + k) * C + j];
                    if (isnan(uv.x)) continue;
                    const long long g = K.pt_off + wk.corr_sp[out_base + i];
                    double p0x, p0y, p0z;
                    xform(c.R, c.t, (double)pk.px[g], (double)pk.py[g], (double)pk.pz[g], p0x, p0y, p0z);
                    const double p1x = dadd(dot3e((double)rp[0], (double)rp[1], (double)rp[2], p0x, p0y, p0z), dmul((double)rp[3], c.s));
                    const double p1y = dadd(dot3e((double)rp[4], (double)rp[5], (double)rp[6], p0x, p0y, p0z), dmul((double)rp[7], c.s));
                    const double p1z = dadd(dot3e((double)rp[8], (double)rp[9], (double)rp[10], p0x, p0y, p0z), dmul((double)rp[11], c.s));
                    const double ou = dadd(ddiv(dmul(fx, p1x), p1z), cx);
                    const double ov = dadd(ddiv(dmul(fy, p1y), p1z), cy);
                    if (!(ou >= 0 && ou < W && ov >= 0 && ov < H)) continue;
                    const double du = dsub(ou, (double)uv.x), dv = dsub(ov, (double)uv.y);
                    const double dist = sqrt(dadd(dmul(du, du), dmul(dv, dv)));
                    if (dist < pr.thr2d) { s2d[h] += dist; v2d[h] += 1.0; }
                    c2d[h] += 1.0;
                }
            }
        }
    }
    // fixed-order block reduction (deterministic): warp w holds the one-kernel K1's warps w (h = 0) and w + 8 (h = 1)
    for (int h = 0; h < 2; ++h) {
        for (int o = 16; o; o >>= 1) {
            s2d[h] += __shfl_down_sync(0xffffffffu, s2d[h], o);
            v2d[h] += __shfl_down_sync(0xffffffffu, v2d[h], o);
            c2d[h] += __shfl_down_sync(0xffffffffu, c2d[h], o);
        }
        if (lane == 0) {
            const int w = warp + h * (kCorrThreads / 32);
            S.red[0][w] = s2d[h]; S.red[1][w] = v2d[h]; S.red[2][w] = c2d[h];
        }
    }
    __syncthreads();
    if (tid == 0) {
        FrameRec r;
        r.s2d = r.v2d = r.c2d = 0;
        for (int w = 0; w < kTermLanes / 32; ++w) { r.s2d += S.red[0][w]; r.v2d += S.red[1][w]; r.c2d += S.red[2][w]; }
        r.she = 0; r.che = 0;
        if (kept && K.he_valid && with_terms) { r.she = S.he_val; r.che = 1; }
        r.kept = kept ? 1.0 : 0.0;
        r.ncorr = kept ? (double)ncorr : 0.0;
        r.nq = kept ? (double)nq : 0.0;
        wk.frame[urec] = r;
        wk.n_corr[urec] = ncorr;
        wk.n_q[urec] = kept ? nq : 0;
    }
}

}  // namespace

size_t assoc2d_split_smem_bytes(int max_band_words, int max_groups) {
    return ((sizeof(StreamSmem) + 15) & ~size_t(15)) + (size_t)max_band_words * 4 + (size_t)kLocalSurv * 4 + 2 * (size_t)max_groups + 16;
}

cudaError_t assoc2d_split_configure(size_t smem) {
    static size_t granted[64] = {0};
    static std::mutex mu;
    std::lock_guard<std::mutex> lk(mu);
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
    if (smem <= granted[dev] || smem <= 48 * 1024) return cudaSuccess;
    e = cudaFuncSetAttribute(k_stream, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) granted[dev] = smem;
    return e;
}

cudaError_t launch_assoc2d_split(const DevPack &pk, const DevWork &wk, const DevParams &pr, int B, size_t smem, int max_bands, int max_surv_cap,
                                 cudaStream_t st, int with_terms) {
    if (B <= 0 || pk.n_ov_sel <= 0) return cudaSuccess;
    const long long units = (long long)pk.n_ov_sel * B;  // unit = oversize selection position * B + candidate
    // per-unit counters and the per-keypoint tables (indexed by oversize ordinal) start empty (all-ones = "no value": larger
    // than any distance / key)
    cudaError_t e = cudaMemsetAsync(wk.k1_cnt, 0, sizeof(UnitCnt) * (size_t)pk.n_ov * B, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(wk.k1_best_d2, 0xff, 8 * (size_t)pk.n_ov_kp * B, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(wk.k1_best_key, 0xff, 8 * (size_t)pk.n_ov_kp * B, st);
    if (e != cudaSuccess) return e;
    // few (unit, band) pairs (a keyframe shard of a multi-GPU run, one candidate): more CTAs per pair keep the SMs busy
    const long long ub = units * max_bands;
    int S_sub = 2;
    while (S_sub < 8 && ub * S_sub < 148 * 6 * 2) S_sub *= 2;
    if (const char *e2 = getenv("STL_K1_SUB")) S_sub = max(1, min(8, atoi(e2)));  // diagnostic
    if (ub * S_sub > 0x7fffffffll) return cudaErrorInvalidValue;
    k_stream<<<(unsigned)(ub * S_sub), kStreamThreads, smem, st>>>(pk, wk, B, S_sub, max_bands);
    // survivors are 1-2 % of the points: four chunks of 256 threads cover the usual unit (kK1SurvCap), one more per
    // 1024 survivor slots the larger ones, the loop the rest
    const int ychunks = max(4, min(32, (max_surv_cap + 1023) / 1024));
    k_exact<<<dim3((unsigned)units, ychunks), kExactThreads, 0, st>>>(pk, wk, pr, B);
    k_corr<<<(unsigned)units, kCorrThreads, 0, st>>>(pk, wk, pr, B, with_terms);
    return cudaGetLastError();
}

}  // namespace stl
