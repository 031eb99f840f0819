"""The host decisions of a pack upload (csrc/packlayout.hpp) without a GPU: validation, the K1 routing rule with an injected
shared-memory model and limit, the oversize keyframes' workspace slices, the routing of keyframe selections and the invariants
of the K1 tables.  The module and a small driver are built with nvcc as host code (common.cuh defines device helpers beside
its layout structs) and run here; no device and no library is involved."""
import os
import shutil
import subprocess

import pytest

from conftest import PKG

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, PKG, "csrc")

DRIVER = r"""
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>
#include "packlayout.hpp"
using namespace stl;

static int failures = 0;
static void report(const char *name, bool ok, const std::string &why = "") {
    std::printf("%s %s%s\n", name, ok ? "ok" : "FAIL ", ok ? "" : why.c_str());
    failures += !ok;
}

// A pack of keyframes (W, H, keypoints, scan points); keypoints at deterministic pseudo-random pixels, every third without a
// map point; map points at depth 10 along the keypoint's ray with Tcw = [I | 0], so that variant 1 re-projects them onto it
struct Kf { int W, H, n_kp; long long n_pts; };
struct HostPack {
    std::vector<int64_t> scan_off, kp_off;
    std::vector<float> xyz, kp_xy, kp_mp, intr, Tcw, he_Tc;
    std::vector<double> he_Tl;
    std::vector<int32_t> wh;
    std::vector<uint8_t> he_valid;
    stl_pack_t p;
    explicit HostPack(const std::vector<Kf> &kfs) {
        const int F = (int)kfs.size();
        scan_off.assign(1, 0); kp_off.assign(1, 0);
        unsigned s = 7;
        auto rnd = [&]() { s = s * 1664525u + 1013904223u; return (s >> 8) / 16777216.0; };
        for (int f = 0; f < F; ++f) {
            const Kf &k = kfs[f];
            scan_off.push_back(scan_off.back() + k.n_pts); kp_off.push_back(kp_off.back() + k.n_kp);
            const double fx = 0.8 * k.W, fy = 0.75 * k.W, cx = k.W / 2.0, cy = k.H / 2.0;
            intr.insert(intr.end(), {(float)fx, (float)fy, (float)cx, (float)cy});
            wh.insert(wh.end(), {k.W, k.H});
            for (int i = 0; i < k.n_kp; ++i) {
                // corners and borders now and then, to reach the clamped grid cells and the bitmap apron
                double u = rnd() * k.W, v = rnd() * k.H;
                if (i % 17 == 3) { u = 0.0; v = k.H - 0.01; }
                kp_xy.insert(kp_xy.end(), {(float)u, (float)v});
                const float z = 10.f;
                if (i % 3 == 2) kp_mp.insert(kp_mp.end(), {NAN, NAN, NAN});
                else kp_mp.insert(kp_mp.end(), {(float)((u - cx) / fx * z), (float)((v - cy) / fy * z), z});
            }
            const float T[12] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0};
            Tcw.insert(Tcw.end(), T, T + 12); he_Tc.insert(he_Tc.end(), T, T + 12); he_Tl.insert(he_Tl.end(), T, T + 12);
            he_valid.push_back(1);
        }
        xyz.assign(3, 0.f);  // never read by the layout
        memset(&p, 0, sizeof(p));
        p.n_kf = F; p.n_covis = 0;
        p.scan_offset = scan_off.data(); p.scan_xyz = xyz.data();
        p.kp_offset = kp_off.data(); p.kp_xy = kp_xy.data(); p.kp_mappoint = kp_mp.data();
        p.intrinsics = intr.data(); p.image_wh = wh.data(); p.Tcw = Tcw.data();
        p.he_Tc = he_Tc.data(); p.he_Tl = he_Tl.data(); p.he_valid = he_valid.data();
    }
};

// shared-memory models: "own need = keypoints + 1000 per 128-point group" for the routing, a constant for the stream kernel
static size_t smem_kp_groups(int kp, int, int groups) { return (size_t)kp + 1000 * (size_t)groups; }
static size_t smem_split_small(int, int) { return 100; }
static size_t smem_split_large(int, int) { return 1 << 20; }

static K1Limits limits(int optin, bool allow, bool route_all = false) {
    K1Limits l;
    l.smem_optin = optin; l.k1_smem = smem_kp_groups; l.split_smem = smem_split_small; l.allow_oversize = allow; l.route_all = route_all;
    return l;
}
static std::vector<int> ov_of(const PackLayout &L) { std::vector<int> v; for (const OvKf &o : L.ov) v.push_back(o.f); return v; }
static std::string str(const std::vector<int> &v) { std::string s = "["; for (int x : v) s += std::to_string(x) + ","; return s + "]"; }

static void routing_rule() {
    // own needs 100, 400, 200, 300 against 250: 400 and 300 leave, the rest's maximum 200 fits
    HostPack hp({{640, 480, 100, 0}, {640, 480, 400, 0}, {640, 480, 200, 0}, {640, 480, 300, 0}});
    PackLayout L; std::string err;
    stl_status_t s = layout_pack(&hp.p, limits(250, true), L, err);
    report("largest_first", s == STL_OK && ov_of(L) == std::vector<int>{1, 3} && L.n_fit == 2 && L.max_kp == 200 && L.k1_smem == 200 &&
           L.ov_ord == std::vector<int>{-1, 0, -1, 1}, str(ov_of(L)) + " n_fit " + std::to_string(L.n_fit));
    s = layout_pack(&hp.p, limits(250, false), L, err);
    report("refused_without_flag", s == STL_ERR_CAPACITY && err == "K1 needs 400 B of shared memory (400 keypoints); device limit 250", err);
    s = layout_pack(&hp.p, limits(1000, false), L, err);
    report("fits", s == STL_OK && L.ov.empty() && L.n_fit == 4 && L.k1_smem == 400 && L.k1_split_smem == 0, str(ov_of(L)));
    s = layout_pack(&hp.p, limits(1000, false, true), L, err);
    report("route_all", s == STL_OK && ov_of(L) == std::vector<int>{0, 1, 2, 3} && L.n_fit == 0 && L.k1_smem == 0 && L.k1_split_smem == 100,
           str(ov_of(L)));
    K1Limits big = limits(250, true);
    big.split_smem = smem_split_large;
    s = layout_pack(&hp.p, big, L, err);
    report("split_refused", s == STL_ERR_CAPACITY && err == "K1a needs 1048576 B of shared memory; device limit 250", err);
    // a tie of own needs (1200 = 200 + 1000 = 1200 + 0) goes to the lower index: A then B leave (the rest, C, needs 1100);
    // with B first, B alone leaves (the rest's maxima, 200 keypoints and 1 group, need 1200)
    const Kf A{640, 480, 200, 128}, B{640, 480, 1200, 0}, Cc{640, 480, 100, 128};
    HostPack ab({A, B, Cc}), ba({B, A, Cc});
    s = layout_pack(&ab.p, limits(1250, true), L, err);
    report("tie_lower_index_a", s == STL_OK && ov_of(L) == std::vector<int>{0, 1} && L.k1_smem == 1100, str(ov_of(L)));
    s = layout_pack(&ba.p, limits(1250, true), L, err);
    report("tie_lower_index_b", s == STL_OK && ov_of(L) == std::vector<int>{0} && L.k1_smem == 1200, str(ov_of(L)));
}

static void oversize_slices() {
    // 4K landscape / portrait (17 bands of 67 / 120 rows), 1241 x 376 (one band), different survivor caps
    HostPack hp({{3840, 2160, 3000, 10000}, {1241, 376, 100, 128}, {2160, 3840, 5000, 7000}});
    PackLayout L; std::string err;
    const stl_status_t s = layout_pack(&hp.p, limits(1 << 30, true, true), L, err);
    bool ok = s == STL_OK && L.ov.size() == 3;
    const int surv[3] = {6144, 4096, 7040}, bands[3] = {17, 1, 17};
    long long kp = 0, sv = 0, mt = 0;
    for (int i = 0; ok && i < 3; ++i) {
        const OvKf &o = L.ov[i];
        ok = o.f == i && o.surv_cap == surv[i] && o.match_cap == 2 * surv[i] && o.n_bands == bands[i] && o.kp_off == kp && o.surv_off == sv &&
             o.match_off == mt;
        kp += L.kf[i].n_kp; sv += o.surv_cap; mt += o.match_cap;
    }
    ok = ok && L.n_ov_kp == 8100 && L.n_ov_surv == 6144 + 4096 + 7040 && L.n_ov_match == 2 * L.n_ov_surv && L.ov_max_bands == 17 &&
         L.ov_max_surv == 7040;
    report("ovkf_slices", ok);
}

static void selections() {
    // one 128-point group each: own needs 1100, 1400, 1200, 1300, 1030 against 1250, so keyframes 1 and 3 are oversize
    HostPack hp({{640, 480, 100, 10}, {640, 480, 400, 50}, {640, 480, 200, 90}, {640, 480, 300, 110}, {640, 480, 30, 128}});
    PackLayout L; std::string err;
    if (layout_pack(&hp.p, limits(1250, true), L, err) != STL_OK || ov_of(L) != std::vector<int>{1, 3}) { report("selection_setup", false, err); return; }
    auto check = [&](const char *name, const int *kf, int n, const std::vector<int> &fit, const std::vector<int> &ov) {
        const KfRoute r = route_keyframes(L, kf, n);
        const int F = L.n_kf;
        std::vector<int> list(kf ? kf : nullptr, kf ? kf + n : nullptr);
        if (!kf) for (int f = 0; f < F; ++f) list.push_back(f);
        bool ok = r.all == !kf && r.n_sel == (int)list.size() && r.n_fit == (int)fit.size() && r.n_ov == (int)ov.size();
        ok = ok && std::vector<int>(r.lists.begin(), r.lists.begin() + r.n_fit) == fit &&
             std::vector<int>(r.lists.begin() + F, r.lists.begin() + F + r.n_ov) == ov;
        long long pts = 0, kps = 0, slots = 0;
        std::vector<uint8_t> mask(F, 0);
        for (size_t i = 0; i < list.size(); ++i) {
            const DevKf &K = L.kf[list[i]];
            if (kf) ok = ok && r.sel_mp[i].x == slots && r.sel_mp[i].x + r.sel_mp[i].y == K.mp_off;
            pts += K.n_pts; kps += K.n_kp; slots += K.n_mp; mask[list[i]] = 1;
        }
        ok = ok && r.pts == pts && r.kp == kps && r.n_sel_mp == slots && r.mask == mask;
        ok = ok && (kf ? r.sel == list && (int)r.sel_mp.size() == n + 1 && r.sel_mp[n].x == slots : r.sel.empty() && r.sel_mp.empty());
        report(name, ok, "fit " + str(std::vector<int>(r.lists.begin(), r.lists.begin() + r.n_fit)) + " ov " +
                         str(std::vector<int>(r.lists.begin() + F, r.lists.begin() + F + r.n_ov)));
    };
    static const int none[1] = {0}, fitting[3] = {0, 2, 4}, oversize[2] = {1, 3}, mixed[3] = {0, 3, 4};
    check("route_all_keyframes", nullptr, 0, {0, 2, 4}, {0, 1});
    check("route_empty", none, 0, {}, {});
    check("route_only_fitting", fitting, 3, {0, 2, 4}, {});
    check("route_only_oversize", oversize, 2, {}, {0, 1});
    check("route_mixed", mixed, 3, {0, 4}, {1});
}

static void validation() {
    const K1Limits lim = limits(1 << 30, false);
    PackLayout L; std::string err;
    auto expect = [&](const char *name, HostPack &hp, stl_status_t code, const char *msg) {
        err.clear();
        const stl_status_t s = layout_pack(&hp.p, lim, L, err);
        report(name, s == code && err == msg, std::to_string(s) + " " + err);
    };
    { HostPack hp({{640, 480, 10, 100}}); hp.p.n_kf = 0; expect("bad_n_kf", hp, STL_ERR_INVALID, "bad n_kf/n_covis"); }
    { HostPack hp({{640, 480, 10, 100}}); hp.p.image_wh = nullptr; expect("null_member", hp, STL_ERR_INVALID, "null pack member"); }
    { HostPack hp({{640, 480, 10, 100}}); hp.kp_off[0] = 1; expect("offsets_start", hp, STL_ERR_INVALID, "offsets must start at 0"); }
    { HostPack hp({{640, 480, 10, 100}, {640, 480, 10, 100}}); hp.scan_off[2] = 50;
      expect("non_monotone_offsets", hp, STL_ERR_INVALID, "offsets must be non-decreasing (keyframe 1)"); }
    { HostPack hp({{640, 480, 10, 100}}); hp.p.kp_xy = nullptr; expect("null_kp_xy", hp, STL_ERR_INVALID, "kp_xy / kp_mappoint is null"); }
    { HostPack hp({{640, 480, 10, 100}}); hp.p.n_covis = 1;
      expect("null_covis", hp, STL_ERR_INVALID, "covis_relpose / covis_valid / covis_uv is null although n_covis > 0"); }
    { HostPack hp({{640, 480, 10, 1048577}}); expect("scan_too_large", hp, STL_ERR_CAPACITY, "scan 0 has 1048577 points (limit 1048576)"); }
    { HostPack hp({{640, 480, 10, 100}, {0, 480, 10, 100}}); expect("bad_image_size", hp, STL_ERR_INVALID, "bad image size of keyframe 1"); }
    { HostPack hp({{640, 480, 10, 100}, {16385, 480, 10, 100}}); expect("image_too_wide", hp, STL_ERR_INVALID, "bad image size of keyframe 1"); }
    { HostPack hp({{640, 480, 65536, 100}}); expect("too_many_keypoints", hp, STL_ERR_CAPACITY, "more than 65535 keypoints in a keyframe"); }
}

static int a16(int x) { return (x + 15) / 16 * 16; }

static void tables(int W, int H, int variant) {
    const std::string tag = std::to_string(W) + "x" + std::to_string(H) + "_v" + std::to_string(variant);
    HostPack hp({{W, H, 3000, 4000}, {W, H, 0, 128}, {W, H, 700, 4000}});
    PackLayout L; std::string err;
    const double mpd = 1.5;
    if (layout_pack(&hp.p, limits(1 << 30, false), L, err) != STL_OK) { report(("tables_" + tag).c_str(), false, err); return; }
    PackTables t;
    build_tables(&hp.p, L, variant, mpd, t);
    bool grid = true, bitmap = true, blob = true, pixels = true;
    long long tab = 0;
    for (int f = 0; f < L.n_kf; ++f) {
        const DevKf &K = L.kf[f];
        const int ncell = K.gw * K.gh, n = K.n_kp;
        const float *q = t.kp_xy + 2 * K.kp_off;
        // query pixels: the pack's, or under variant 1 the re-projected map points (NaN without one) and their float32 copy
        for (int k = 0; k < n; ++k) {
            const float *mp = hp.kp_mp.data() + 3 * (K.kp_off + k);
            if (variant == 0) { pixels &= q[2 * k] == hp.kp_xy[2 * (K.kp_off + k)] && q[2 * k + 1] == hp.kp_xy[2 * (K.kp_off + k) + 1]; continue; }
            const double *d = t.kp_xyd.data() + 2 * (K.kp_off + k);
            if (std::isnan(mp[0])) { pixels &= std::isnan(d[0]) && std::isnan(d[1]) && std::isnan(q[2 * k]); continue; }
            pixels &= std::fabs(d[0] - hp.kp_xy[2 * (K.kp_off + k)]) < 1e-3 && std::fabs(d[1] - hp.kp_xy[2 * (K.kp_off + k) + 1]) < 1e-3 &&
                      q[2 * k] == (float)d[0] && q[2 * k + 1] == (float)d[1];
        }
        // grid_kp: a permutation of the keyframe's keypoints bucketed by 8 px cell (clamped; unqueried ones in cell 0);
        // grid_start: its prefix
        const uint32_t *gs = t.grid_start.data() + K.grid_off, *gk = t.grid_kp.data() + K.kp_off;
        std::vector<int> seen(n, 0), count(ncell, 0), cell(n, 0);
        for (int k = 0; k < n; ++k) {
            const double x = q[2 * k], y = q[2 * k + 1];
            int cx = 0, cy = 0;
            if (x == x && y == y) { cx = std::min(std::max((int)std::floor(x / 8), 0), K.gw - 1); cy = std::min(std::max((int)std::floor(y / 8), 0), K.gh - 1); }
            cell[k] = cy * K.gw + cx;
            ++count[cell[k]];
        }
        grid &= gs[0] == 0 && (int)gs[ncell] == n;
        for (int c = 0; c < ncell && grid; ++c) {
            grid &= (int)(gs[c + 1] - gs[c]) == count[c];
            for (uint32_t i = gs[c]; i < gs[c + 1] && grid; ++i) grid &= gk[i] < (uint32_t)n && !seen[gk[i]]++ && cell[gk[i]] == c;
        }
        // bitmap: every 2 px cell (1-cell apron) with a point closer than max_pixel_dist + kFastErrPx to a query pixel is set
        const uint32_t *bm = t.bitmap.data() + K.bm_off;
        const double R = mpd + kFastErrPx;
        for (int k = 0; k < n && bitmap; ++k) {
            const double x = variant == 1 ? t.kp_xyd[2 * (K.kp_off + k)] : q[2 * k], y = variant == 1 ? t.kp_xyd[2 * (K.kp_off + k) + 1] : q[2 * k + 1];
            if (!(x == x)) continue;
            const int c0 = std::max(0, (int)std::floor((x - R) / 2)), c1 = (int)std::floor((x + R) / 2) + 1;
            const int r0 = std::max(0, (int)std::floor((y - R) / 2)), r1 = (int)std::floor((y + R) / 2) + 1;
            for (int r = r0; r <= r1 && bitmap; ++r)
                for (int c = c0; c <= c1; ++c) {
                    const double x0 = 2.0 * (c - 1), y0 = 2.0 * (r - 1);  // the cell covers [x0, x0 + 2) x [y0, y0 + 2)
                    const double dx = std::max({x0 - x, x - (x0 + 2), 0.0}), dy = std::max({y0 - y, y - (y0 + 2), 0.0});
                    if (dx * dx + dy * dy >= R * R || c > (W + 1) / 2 + 1 || r > (H + 1) / 2 + 1) continue;
                    if (!((bm[r * K.bm_wpr + (c >> 5)] >> (c & 31)) & 1u)) { bitmap = false; break; }
                }
        }
        // k1tab: [float2 kp[n]] [uint32 bitmap] [uint16 grid_start[ncell + 1]] [uint16 grid_kp[n]] [uint32 has_mp[(n + 31) / 32]],
        // each section 16-byte aligned and zero-padded
        const int words = K.bm_wpr * K.bm_rows;
        std::vector<uint8_t> want(a16(8 * n) + a16(4 * words) + a16(2 * (ncell + 1)) + a16(2 * n) + a16(4 * ((n + 31) / 32)), 0);
        uint8_t *w = want.data();
        memcpy(w, q, 8 * (size_t)n); w += a16(8 * n);
        memcpy(w, bm, 4 * (size_t)words); w += a16(4 * words);
        for (int i = 0; i <= ncell; ++i) { const uint16_t v = (uint16_t)gs[i]; memcpy(w + 2 * i, &v, 2); }
        w += a16(2 * (ncell + 1));
        for (int k = 0; k < n; ++k) { const uint16_t v = (uint16_t)gk[k]; memcpy(w + 2 * k, &v, 2); }
        w += a16(2 * n);
        for (int k = 0; k < n; ++k) if (!std::isnan(hp.kp_mp[3 * (K.kp_off + k)])) w[k / 8] |= (uint8_t)(1u << (k % 8));
        blob &= K.tab_off == tab && K.tab_bytes == (int)want.size() && memcmp(t.k1tab.data() + K.tab_off, want.data(), want.size()) == 0;
        tab += K.tab_bytes;
    }
    report(("query_pixels_" + tag).c_str(), pixels);
    report(("grid_" + tag).c_str(), grid);
    report(("bitmap_" + tag).c_str(), bitmap);
    report(("k1tab_" + tag).c_str(), blob && (long long)t.k1tab.size() == std::max(tab, 16ll));
}

int main() {
    routing_rule();
    oversize_slices();
    selections();
    validation();
    for (int variant = 0; variant < 2; ++variant) { tables(1241, 376, variant); tables(333, 251, variant); }
    return failures;
}
"""

CHECKS = (["largest_first", "refused_without_flag", "fits", "route_all", "split_refused", "tie_lower_index_a", "tie_lower_index_b",
           "ovkf_slices", "route_all_keyframes", "route_empty", "route_only_fitting", "route_only_oversize", "route_mixed",
           "bad_n_kf", "null_member", "offsets_start", "non_monotone_offsets", "null_kp_xy", "null_covis", "scan_too_large",
           "bad_image_size", "image_too_wide", "too_many_keypoints"] +
          [f"{what}_{wh}_v{v}" for v in (0, 1) for wh in ("1241x376", "333x251") for what in ("query_pixels", "grid", "bitmap", "k1tab")])


@pytest.fixture(scope="module")
def results(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    d = tmp_path_factory.mktemp("packlayout")
    src, exe = d / "driver.cpp", d / "driver"
    src.write_text(DRIVER)
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O1", "-ccbin", "/usr/bin/g++", "-Xcompiler", "-fopenmp", "-I" + CSRC, "-x", "cu",
           str(src), os.path.join(CSRC, "packlayout.cpp"), "-o", str(exe)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-4000:]
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    out = {}
    for line in r.stdout.splitlines():
        name, _, rest = line.partition(" ")
        out[name] = rest
    return out


@pytest.mark.parametrize("check", CHECKS)
def test_pack_layout(results, check):
    assert results.get(check) == "ok", f"{check}: {results.get(check, 'not reported')}"
