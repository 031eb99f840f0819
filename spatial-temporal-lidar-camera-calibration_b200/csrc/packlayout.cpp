// packlayout.cpp — see packlayout.hpp.  Host code only (built with nvcc -x cu for common.cuh).
#include "packlayout.hpp"

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>

namespace stl {

namespace {

stl_status_t fail(std::string &err, stl_status_t code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    err = buf;
    return code;
}

}  // namespace

stl_status_t layout_pack(const stl_pack_t *p, const K1Limits &lim, PackLayout &L, std::string &err) {
    if (p->n_kf <= 0 || p->n_covis < 0 || p->n_covis > STL_MAX_COVIS) return fail(err, STL_ERR_INVALID, "bad n_kf/n_covis");
    if (!p->scan_offset || !p->kp_offset || !p->intrinsics || !p->image_wh || !p->Tcw || !p->he_Tc || !p->he_Tl || !p->he_valid)
        return fail(err, STL_ERR_INVALID, "null pack member");
    const int F = p->n_kf, C = p->n_covis;
    if (p->scan_offset[0] != 0 || p->kp_offset[0] != 0) return fail(err, STL_ERR_INVALID, "offsets must start at 0");
    for (int f = 0; f < F; ++f)
        if (p->scan_offset[f + 1] < p->scan_offset[f] || p->kp_offset[f + 1] < p->kp_offset[f])
            return fail(err, STL_ERR_INVALID, "offsets must be non-decreasing (keyframe %d)", f);
    if (p->scan_offset[F] > (1ll << 40) || p->kp_offset[F] > (1ll << 31))
        return fail(err, STL_ERR_CAPACITY, "pack too large (%lld points, %lld keypoints)", (long long)p->scan_offset[F], (long long)p->kp_offset[F]);
    if (p->scan_offset[F] > 0 && !p->scan_xyz) return fail(err, STL_ERR_INVALID, "scan_xyz is null");
    if (p->kp_offset[F] > 0 && (!p->kp_xy || !p->kp_mappoint)) return fail(err, STL_ERR_INVALID, "kp_xy / kp_mappoint is null");
    if (C > 0 && (!p->covis_relpose || !p->covis_valid || (p->kp_offset[F] > 0 && !p->covis_uv)))
        return fail(err, STL_ERR_INVALID, "covis_relpose / covis_valid / covis_uv is null although n_covis > 0");

    // ---- per-keyframe metadata
    L = PackLayout();
    L.n_kf = F; L.n_covis = C;
    std::vector<DevKf> &hk = L.kf;
    hk.assign(F, DevKf());
    long long pt = 0, nodes = 0, bmw = 0, gcells = 0, mp_total = 0, tab_total = 0;
    int max_kp = 0, max_tab = 0;
    for (int f = 0; f < F; ++f) {
        DevKf &K = hk[f];
        const long long n = p->scan_offset[f + 1] - p->scan_offset[f];
        const long long nk = p->kp_offset[f + 1] - p->kp_offset[f];
        if (n > (1 << 20)) return fail(err, STL_ERR_CAPACITY, "scan %d has %lld points (limit 1048576)", f, n);
        K.n_pts = (int)n;
        K.n_pad = (int)((n + kPadPts - 1) / kPadPts * kPadPts);
        const int nleaf = K.n_pad / kLeaf;
        K.n0 = std::max(32, (nleaf + 31) / 32 * 32);
        K.n1 = std::max(32, (K.n0 / 32 + 31) / 32 * 32);
        K.n2 = K.n1 / 32;
        K.pt_off = pt; pt += K.n_pad;
        K.node_off = nodes; nodes += K.n0 + K.n1 + 32;
        K.kp_off = p->kp_offset[f];
        K.n_kp = (int)nk;
        K.fx = p->intrinsics[f * 4]; K.fy = p->intrinsics[f * 4 + 1]; K.cx = p->intrinsics[f * 4 + 2]; K.cy = p->intrinsics[f * 4 + 3];
        K.W = p->image_wh[f * 2]; K.H = p->image_wh[f * 2 + 1];
        if (K.W <= 0 || K.H <= 0 || K.W > 16384 || K.H > 16384) return fail(err, STL_ERR_INVALID, "bad image size of keyframe %d", f);
        const int bw_total = (K.W + kBmCell - 1) / kBmCell + 2;
        K.bm_wpr = (bw_total + 1 + 31) / 32;
        K.bm_rows = (K.H + kBmCell - 1) / kBmCell + 3;
        K.bm_off = bmw; bmw += (long long)K.bm_wpr * K.bm_rows;
        K.gw = std::max(1, (K.W + kGridCell - 1) / kGridCell);
        K.gh = std::max(1, (K.H + kGridCell - 1) / kGridCell);
        K.grid_off = gcells; gcells += (long long)K.gw * K.gh + 1;
        {
            const K1Tab tl = k1tab_layout(K.n_kp, K.bm_wpr * K.bm_rows, K.gw * K.gh);
            K.tab_off = tab_total; K.tab_bytes = tl.bytes; tab_total += tl.bytes;
            max_tab = std::max(max_tab, tl.bytes);
        }
        K.he_valid = p->he_valid[f] ? 1 : 0;
        K.covis_mask = 0;
        for (int j = 0; j < C; ++j) K.covis_mask |= (p->covis_valid[(size_t)f * C + j] ? 1u : 0u) << j;
        K.mp_off = mp_total;
        K.n_mp = 0;
        for (long long k = 0; k < nk; ++k) K.n_mp += !(p->kp_mappoint[(K.kp_off + k) * 3] != p->kp_mappoint[(K.kp_off + k) * 3]);
        mp_total += K.n_mp;
        K.pmax = 1.f;
        max_kp = std::max(max_kp, K.n_kp);
    }
    L.n_pad_total = pt; L.n_nodes_total = nodes; L.n_kp_total = p->kp_offset[F]; L.n_mp_total = mp_total;
    L.bm_words = bmw; L.grid_cells = gcells; L.tab_bytes = tab_total;
    int max_groups = 0;
    for (int f = 0; f < F; ++f) max_groups = std::max(max_groups, hk[f].n_pad / 128);
    if (max_kp > 65535) return fail(err, STL_ERR_CAPACITY, "more than 65535 keypoints in a keyframe");

    // ---- K1 routing (stlcalib.h, stl_allow_oversize_keyframes); with no keyframe out this is the check of a pack without
    // oversize keyframes
    std::vector<int> order(F);
    std::vector<size_t> own(F);
    for (int f = 0; f < F; ++f) { order[f] = f; own[f] = lim.k1_smem(hk[f].n_kp, hk[f].tab_bytes, hk[f].n_pad / 128); }
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return own[a] > own[b]; });
    std::vector<int> sfx_kp(F + 1, 0), sfx_tab(F + 1, 0), sfx_gr(F + 1, 0);  // maxima over order[r..F)
    for (int r = F - 1; r >= 0; --r) {
        const DevKf &K = hk[order[r]];
        sfx_kp[r] = std::max(sfx_kp[r + 1], K.n_kp); sfx_tab[r] = std::max(sfx_tab[r + 1], K.tab_bytes); sfx_gr[r] = std::max(sfx_gr[r + 1], K.n_pad / 128);
    }
    int n_out = 0;
    while (n_out < F && lim.k1_smem(sfx_kp[n_out], sfx_tab[n_out], sfx_gr[n_out]) > (size_t)lim.smem_optin) ++n_out;
    if (n_out > 0 && !lim.allow_oversize)
        return fail(err, STL_ERR_CAPACITY, "K1 needs %zu B of shared memory (%d keypoints); device limit %d", lim.k1_smem(max_kp, max_tab, max_groups),
                    max_kp, lim.smem_optin);
    if (lim.route_all) n_out = F;
    L.n_fit = F - n_out;
    L.max_kp = sfx_kp[n_out]; L.max_tab = sfx_tab[n_out]; L.max_groups = sfx_gr[n_out];
    if (L.n_fit > 0) L.k1_smem = lim.k1_smem(L.max_kp, L.max_tab, L.max_groups);
    // the oversize keyframes, increasing, and their workspace slices
    L.ov_ord.assign(F, -1);
    for (int r = 0; r < n_out; ++r) L.ov_ord[order[r]] = 0;
    int ov_band_words = 0, ov_groups = 0;
    for (int f = 0; f < F; ++f) {
        if (L.ov_ord[f] < 0) continue;
        L.ov_ord[f] = (int)L.ov.size();
        const DevKf &K = hk[f];
        OvKf o;
        o.f = f;
        o.surv_cap = (int)std::max<long long>(kK1SurvCap, std::min<long long>(((2ll * K.n_kp + 255) / 256) * 256, K.n_pad));
        o.match_cap = 2 * o.surv_cap;
        const int rows = k1_band_rows(K.bm_wpr);
        o.n_bands = (K.bm_rows + rows - 1) / rows;
        o.kp_off = L.n_ov_kp; o.surv_off = L.n_ov_surv; o.match_off = L.n_ov_match;
        L.n_ov_kp += K.n_kp; L.n_ov_surv += o.surv_cap; L.n_ov_match += o.match_cap;
        L.ov_max_bands = std::max(L.ov_max_bands, o.n_bands); L.ov_max_surv = std::max(L.ov_max_surv, o.surv_cap);
        ov_band_words = std::max(ov_band_words, std::min(rows, K.bm_rows) * K.bm_wpr); ov_groups = std::max(ov_groups, K.n_pad / 128);
        L.ov.push_back(o);
    }
    if (n_out > 0) {
        L.k1_split_smem = lim.split_smem(ov_band_words, ov_groups);
        if (L.k1_split_smem > (size_t)lim.smem_optin)
            return fail(err, STL_ERR_CAPACITY, "K1a needs %zu B of shared memory; device limit %d", L.k1_split_smem, lim.smem_optin);
    }
    return STL_OK;
}

void build_tables(const stl_pack_t *p, const PackLayout &L, int variant, double max_pixel_dist, PackTables &t) {
    const int F = L.n_kf;
    const long long NK = L.n_kp_total;
    // ---- variant 1: the fp64 query pixels and their float32 copy (the coarse tables' margins cover its rounding)
    t.kp_xy = p->kp_xy;
    if (variant == 1) {
        t.kp_xyd.assign((size_t)std::max<long long>(NK, 1) * 2, std::nan(""));
        t.kp_xyf.assign((size_t)std::max<long long>(NK, 1) * 2, std::nanf(""));
        double *kpd = t.kp_xyd.data();
        float *kpf = t.kp_xyf.data();
#pragma omp parallel for schedule(static)
        for (int f = 0; f < F; ++f) {
            const float *T = p->Tcw + (size_t)f * 12;
            const double fx = p->intrinsics[f * 4], fy = p->intrinsics[f * 4 + 1], cx = p->intrinsics[f * 4 + 2], cy = p->intrinsics[f * 4 + 3];
            for (long long k = p->kp_offset[f]; k < p->kp_offset[f + 1]; ++k) {
                const float *mp = p->kp_mappoint + k * 3;
                if (mp[0] != mp[0]) continue;
                const double X = mp[0], Y = mp[1], Z = mp[2];
                double P[3];
                for (int i = 0; i < 3; ++i)
                    P[i] = (((double)T[i * 4] * X + (double)T[i * 4 + 1] * Y) + (double)T[i * 4 + 2] * Z) + (double)T[i * 4 + 3];
                kpd[k * 2] = fx * P[0] / P[2] + cx;
                kpd[k * 2 + 1] = fy * P[1] / P[2] + cy;
                kpf[k * 2] = (float)kpd[k * 2];
                kpf[k * 2 + 1] = (float)kpd[k * 2 + 1];
            }
        }
        t.kp_xy = kpf;
    }
    const float *kp_host = t.kp_xy;

    // ---- keypoint bitmap + cell grid
    t.bitmap.assign((size_t)L.bm_words, 0u);
    t.grid_start.assign((size_t)L.grid_cells, 0u);
    t.grid_kp.assign((size_t)std::max<long long>(NK, 1), 0u);
    // variant 1: + the float32 rounding of the coarse keypoint copy (< 1e-3 px for any image size)
    const double Rdil = max_pixel_dist + (double)kFastErrPx + (variant == 1 ? 1e-3 : 0.0);
#pragma omp parallel for schedule(dynamic, 8)
    for (int f = 0; f < F; ++f) {
        const DevKf &K = L.kf[f];
        uint32_t *bm = t.bitmap.data() + K.bm_off;
        uint32_t *gs = t.grid_start.data() + K.grid_off;
        uint32_t *gk = t.grid_kp.data() + K.kp_off;
        const float *kp = kp_host + K.kp_off * 2;
        const int bw_total = (K.W + kBmCell - 1) / kBmCell + 2, bh_total = (K.H + kBmCell - 1) / kBmCell + 2;
        const int ncell = K.gw * K.gh;
        std::vector<uint32_t> cell(K.n_kp);
        for (int k = 0; k < K.n_kp; ++k) {
            const double kx = kp[k * 2], ky = kp[k * 2 + 1];
            int gx = (int)std::floor(kx / kGridCell), gy = (int)std::floor(ky / kGridCell);
            gx = std::min(std::max(gx, 0), K.gw - 1); gy = std::min(std::max(gy, 0), K.gh - 1);
            if (!(kx == kx) || !(ky == ky)) { gx = 0; gy = 0; }
            cell[k] = (uint32_t)(gy * K.gw + gx);
            gs[cell[k] + 1]++;
            if (!(kx == kx) || !(ky == ky)) continue;
            int c0 = (int)std::floor((kx - Rdil) / kBmCell) + 1, c1 = (int)std::floor((kx + Rdil) / kBmCell) + 1;
            int r0 = (int)std::floor((ky - Rdil) / kBmCell) + 1, r1 = (int)std::floor((ky + Rdil) / kBmCell) + 1;
            c0 = std::max(c0, 0); r0 = std::max(r0, 0); c1 = std::min(c1, bw_total - 1); r1 = std::min(r1, bh_total - 1);
            for (int r = r0; r <= r1; ++r)
                for (int cc = c0; cc <= c1; ++cc) bm[r * K.bm_wpr + (cc >> 5)] |= 1u << (cc & 31);
        }
        for (int i = 0; i < ncell; ++i) gs[i + 1] += gs[i];
        std::vector<uint32_t> cur(gs, gs + ncell);
        for (int k = 0; k < K.n_kp; ++k) gk[cur[cell[k]]++] = (uint32_t)k;
    }

    // ---- K1 table blobs: the same tables, per keyframe, contiguous in the order K1 keeps them in shared memory
    t.k1tab.assign((size_t)std::max<long long>(L.tab_bytes, 16), 0);
#pragma omp parallel for schedule(static)
    for (int f = 0; f < F; ++f) {
        const DevKf &K = L.kf[f];
        const int ncell = K.gw * K.gh, bmwords = K.bm_wpr * K.bm_rows;
        const K1Tab tl = k1tab_layout(K.n_kp, bmwords, ncell);
        uint8_t *dst = t.k1tab.data() + K.tab_off;
        memcpy(dst, kp_host + K.kp_off * 2, 8 * (size_t)K.n_kp);
        memcpy(dst + tl.off_bm, t.bitmap.data() + K.bm_off, 4 * (size_t)bmwords);
        uint16_t *gs16 = reinterpret_cast<uint16_t *>(dst + tl.off_gs), *gk16 = reinterpret_cast<uint16_t *>(dst + tl.off_gk);
        uint32_t *mpm = reinterpret_cast<uint32_t *>(dst + tl.off_mp);
        for (int i = 0; i <= ncell; ++i) gs16[i] = (uint16_t)t.grid_start[K.grid_off + i];
        for (int k = 0; k < K.n_kp; ++k) {
            gk16[k] = (uint16_t)t.grid_kp[K.kp_off + k];
            const float m0 = p->kp_mappoint[(K.kp_off + k) * 3];
            if (m0 == m0) mpm[k >> 5] |= 1u << (k & 31);
        }
    }
}

KfRoute route_keyframes(const PackLayout &L, const int *kf, int n) {
    const int F = L.n_kf;
    KfRoute r;
    r.all = kf == nullptr;
    r.n_sel = r.all ? F : n;
    r.mask.assign((size_t)F, r.all ? 1 : 0);
    r.lists.assign((size_t)2 * F, 0);
    if (!r.all) { r.sel.assign(kf, kf + n); r.sel_mp.resize((size_t)n + 1); }
    long long slots = 0;
    for (int i = 0; i < r.n_sel; ++i) {
        const int f = r.all ? i : kf[i];
        const DevKf &K = L.kf[f];
        if (!r.all) { r.sel_mp[i] = make_int2((int)slots, (int)(K.mp_off - slots)); r.mask[f] = 1; }
        slots += K.n_mp; r.pts += K.n_pts; r.kp += K.n_kp;
        if (L.ov_ord[f] >= 0) r.lists[(size_t)F + r.n_ov++] = L.ov_ord[f];
        else r.lists[r.n_fit++] = f;
    }
    if (!r.all) r.sel_mp[n] = make_int2((int)slots, 0);
    r.n_sel_mp = slots;
    return r;
}

}  // namespace stl
