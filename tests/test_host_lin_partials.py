"""The chain-rule rows of k_linearize (csrc/linrow.cuh) against a forward-mode Dual<7> evaluation of the same factors, on the
host (no GPU).  Values are bit-identical.  Partials agree within 1e-13 of the row's largest partial; a 3-D/2-D row whose partials
cancel (the point moves almost along its viewing ray) may differ more, and over those rows the chain rule's largest error
against a long-double evaluation must stay within twice the dual evaluation's."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "spatial-temporal-lidar-camera-calibration_b200", "csrc")

SRC = r"""
#include <cstdio>
#include <cmath>
#include <random>
#include "linrow.cuh"
using namespace stl;

static int fails = 0;
static double worst = 0.0;
static long rows = 0, cancelling = 0;
static double worst_chain = 0.0, worst_dual = 0.0;

// forward-mode dual in long double: the reference for rows whose partials cancel
struct L7 { long double a, v[7]; };
static L7 ld(const D7 &d) { L7 r; r.a = d.a; for (int i = 0; i < 7; ++i) r.v[i] = d.v[i]; return r; }
static L7 lc(double x) { L7 r; r.a = x; for (int i = 0; i < 7; ++i) r.v[i] = 0.0L; return r; }
static L7 operator+(const L7 &f, const L7 &g) { L7 r; r.a = f.a + g.a; for (int i = 0; i < 7; ++i) r.v[i] = f.v[i] + g.v[i]; return r; }
static L7 operator*(const L7 &f, const L7 &g) { L7 r; r.a = f.a * g.a; for (int i = 0; i < 7; ++i) r.v[i] = f.a * g.v[i] + f.v[i] * g.a; return r; }
static L7 operator/(const L7 &f, const L7 &g) { L7 r; r.a = f.a / g.a; for (int i = 0; i < 7; ++i) r.v[i] = (f.v[i] - r.a * g.v[i]) / g.a; return r; }

static void check(const char *what, int blk, const Row7 &r, const D7 &e, const L7 *ref = nullptr) {
    ++rows;
    double big = 0.0, err = 0.0;
    for (int k = 0; k < 7; ++k) { big = std::fmax(big, std::fabs(e.v[k])); err = std::fmax(err, std::fabs(r.v[k] - e.v[k])); }
    const double rel = big > 0.0 ? err / big : err;
    bool ok = rel <= 1e-13;
    if (ok) worst = std::fmax(worst, rel);
    if (!ok && ref) {  // judged in aggregate below, against the long-double evaluation
        long double ec = 0.0L, ed = 0.0L;
        for (int k = 0; k < 7; ++k) { ec = std::fmax(ec, std::fabs(r.v[k] - ref->v[k])); ed = std::fmax(ed, std::fabs(e.v[k] - ref->v[k])); }
        worst_chain = std::fmax(worst_chain, (double)(ec / big));
        worst_dual = std::fmax(worst_dual, (double)(ed / big));
        ok = true;
        ++cancelling;
    }
    if (r.a != e.a || !ok) {
        if (++fails < 10) std::printf("FAIL %s block %d: value %.17g vs %.17g, partial rel err %.3g\n", what, blk, r.a, e.a, rel);
    }
}

static void mv3(const D7 *M, const D7 *p, D7 *o) {
    for (int i = 0; i < 3; ++i) o[i] = (M[i * 3] * p[0] + M[i * 3 + 1] * p[1]) + M[i * 3 + 2] * p[2];
}

int main() {
    std::mt19937_64 rng(12345);
    std::uniform_real_distribution<double> U(-1.0, 1.0);
    const int C = 3;
    for (int cand = 0; cand < 200; ++cand) {
        double x[7];
        const double rs = cand % 4 == 0 ? 1e-5 : 0.3;  // also the small-angle branch of Sim3Exp
        for (int i = 0; i < 3; ++i) x[i] = rs * U(rng);
        for (int i = 3; i < 6; ++i) x[i] = 0.5 * U(rng);
        x[6] = 1.0 + 0.2 * U(rng);
        LmCand c;
        make_lm_candidate(x, &c);
        double W[9][7];
        lin_table(c, W, 0, 1);
        for (int blk = 0; blk < 50; ++blk) {
            // ---- 3-D/3-D: map point, scan point nearby, unit normal
            double g[9];
            for (int i = 0; i < 3; ++i) g[i] = 20.0 * U(rng) + (i == 2 ? 25.0 : 0.0);
            for (int i = 0; i < 3; ++i) g[3 + i] = g[i] + 2.0 * U(rng);
            double nn = 0.0;
            for (int i = 0; i < 3; ++i) { g[6 + i] = U(rng); nn += g[6 + i] * g[6 + i]; }
            for (int i = 0; i < 3; ++i) g[6 + i] /= std::sqrt(nn);
            D7 Ms[3], M[3], d7[3];
            for (int i = 0; i < 3; ++i) Ms[i] = c.s * g[i];
            mv3(c.Rlc, Ms, M);
            for (int i = 0; i < 3; ++i) d7[i] = (M[i] + c.tlc[i]) - g[3 + i];
            double d[3];
            p3_values(c, g, d);
            for (int i = 0; i < 3; ++i) check("point-to-point", blk, p3_point_row(c, W, g, d, i), d7[i]);
            check("point-to-plane", blk, p3_plane_row(c, W, g, d), (d7[0] * g[6] + d7[1] * g[7]) + d7[2] * g[8]);

            // ---- 3-D/2-D: plane point / normal in front of the camera, keypoint ray, C covisible keyframes
            double h[6];
            for (int i = 0; i < 3; ++i) h[i] = 10.0 * U(rng) + (i == 2 ? 20.0 : 0.0);
            nn = 0.0;
            for (int i = 0; i < 3; ++i) { h[3 + i] = 0.2 * U(rng) + (i == 2 ? -1.0 : 0.0); nn += h[3 + i] * h[3 + i]; }
            for (int i = 0; i < 3; ++i) h[3 + i] /= std::sqrt(nn);
            const double fx = 718.856 * (1.0 + 0.05 * U(rng)), fy = fx * (1.0 + 0.03 * U(rng)), cx = 607.19, cy = 185.22;
            const float kx = (float)(607.0 + 300.0 * U(rng)), ky = (float)(185.0 + 180.0 * U(rng));
            const double Cxz = ((double)kx - cx) / fx, Cyz = ((double)ky - cy) / fy;
            const D7 p0[3] = {d7_const(h[0]), d7_const(h[1]), d7_const(h[2])}, n0[3] = {d7_const(h[3]), d7_const(h[4]), d7_const(h[5])};
            D7 p0c[3], n0c[3];
            mv3(c.R, p0, p0c);
            for (int i = 0; i < 3; ++i) p0c[i] = p0c[i] + c.t[i];
            mv3(c.R, n0, n0c);
            const D7 num = (n0c[0] * p0c[0] + n0c[1] * p0c[1]) + n0c[2] * p0c[2];
            const D7 den = (n0c[0] * Cxz + n0c[1] * Cyz) + n0c[2];
            const D7 Z0 = num / den;
            const D7 P0[3] = {Z0 * Cxz, Z0 * Cyz, Z0};
            double z0, dZ[7];
            p2_depth(c, h, Cxz, Cyz, z0, dZ);
            if (z0 != Z0.a) { if (++fails < 10) std::printf("FAIL depth block %d\n", blk); }
            // covisible slots: none, one, or all of them valid
            const int nvalid = blk % 3 == 0 ? 0 : (blk % 3 == 1 ? 1 : C);
            for (int s = 0; s < nvalid; ++s) {
                float rp[12];
                double ang[3] = {0.05 * U(rng), 0.05 * U(rng), 0.05 * U(rng)};
                // small rotation (first order, float) and a forward-biased translation
                const double Rr[9] = {1.0, -ang[2], ang[1], ang[2], 1.0, -ang[0], -ang[1], ang[0], 1.0};
                for (int i = 0; i < 3; ++i) {
                    for (int j = 0; j < 3; ++j) rp[i * 4 + j] = (float)Rr[i * 3 + j];
                    rp[i * 4 + 3] = (float)(i == 2 ? -1.0 - U(rng) : 0.3 * U(rng));
                }
                const float u = (float)(kx + 5.0 * U(rng)), v = (float)(ky + 5.0 * U(rng));
                D7 P1[3];
                for (int i = 0; i < 3; ++i)
                    P1[i] = ((P0[0] * (double)rp[i * 4] + P0[1] * (double)rp[i * 4 + 1]) + P0[2] * (double)rp[i * 4 + 2]) + c.s * (double)rp[i * 4 + 3];
                const D7 eu7 = ((P1[0] * fx) / P1[2] + cx) - (double)u;
                const D7 ev7 = ((P1[1] * fy) / P1[2] + cy) - (double)v;
                double q[3];
                p2_point(c, rp, z0, Cxz, Cyz, q);
                for (int i = 0; i < 3; ++i)
                    if (q[i] != P1[i].a) { if (++fails < 10) std::printf("FAIL P1 block %d\n", blk); }
                Row7 eu, ev;
                p2_rows(c, rp, q, dZ, Cxz, Cyz, fx, fy, cx, cy, u, v, eu, ev);
                L7 Rl[9], tl[3], pc[3], nc[3], Q1[3];
                for (int i = 0; i < 9; ++i) Rl[i] = ld(c.R[i]);
                for (int i = 0; i < 3; ++i) tl[i] = ld(c.t[i]);
                for (int i = 0; i < 3; ++i) {
                    pc[i] = ((Rl[i * 3] * lc(h[0]) + Rl[i * 3 + 1] * lc(h[1])) + Rl[i * 3 + 2] * lc(h[2])) + tl[i];
                    nc[i] = (Rl[i * 3] * lc(h[3]) + Rl[i * 3 + 1] * lc(h[4])) + Rl[i * 3 + 2] * lc(h[5]);
                }
                const L7 Z = ((nc[0] * pc[0] + nc[1] * pc[1]) + nc[2] * pc[2]) / ((nc[0] * lc(Cxz) + nc[1] * lc(Cyz)) + nc[2]);
                const L7 Q0[3] = {Z * lc(Cxz), Z * lc(Cyz), Z};
                for (int i = 0; i < 3; ++i)
                    Q1[i] = ((Q0[0] * lc(rp[i * 4]) + Q0[1] * lc(rp[i * 4 + 1])) + Q0[2] * lc(rp[i * 4 + 2])) + ld(c.s) * lc(rp[i * 4 + 3]);
                const L7 eul = (Q1[0] * lc(fx)) / Q1[2], evl = (Q1[1] * lc(fy)) / Q1[2];
                check("3-D/2-D eu", blk, eu, eu7, &eul);
                check("3-D/2-D ev", blk, ev, ev7, &evl);
            }
        }
    }
    if (worst_chain > 2.0 * worst_dual) ++fails;
    std::printf("rows %ld fails %d worst %.3g; %ld cancelling rows, worst against long double: chain rule %.3g, dual %.3g\n", rows, fails,
                worst, cancelling, worst_chain, worst_dual);
    return fails != 0;
}
"""


def test_chain_rule_rows_match_dual_evaluation(tmp_path):
    src = tmp_path / "lin_partials.cpp"
    exe = tmp_path / "lin_partials"
    src.write_text(SRC)
    r = subprocess.run(["/usr/bin/g++", "-std=c++17", "-O2", "-ffp-contract=off", "-I" + CSRC, str(src), "-o", str(exe)],
                       capture_output=True, text=True)
    if r.returncode != 0:
        pytest.fail("compile failed:\n" + r.stderr[-4000:])
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-4000:]
    assert "rows" in r.stdout and " fails 0 " in r.stdout, r.stdout
