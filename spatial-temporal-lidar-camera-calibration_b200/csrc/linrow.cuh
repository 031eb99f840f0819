// linrow.cuh — residual rows of the frozen plane / point blocks of K4b (k_linearize), host + device.
//
// The VALUES are formed exactly as a forward-mode Dual<7> evaluation of the factor forms them (same operations, same order,
// separate multiply and add), so residuals, costs and the robust-kernel branch do not depend on how the partials are formed.
// The PARTIALS are formed by the chain rule from a few candidate tables instead of carrying seven partials through every
// product: with x = [omega, upsilon, s], only R, t (Sim3Exp(x)), Rlc, tlc (SE3Exp(-x[0:6])) and s depend on x, and every
// block is linear in their entries.  A partial differs from the dual's by a few roundings.
//
//   3-D/3-D (Point2Point / Point2Plane, IBACalib2.hpp:570-584,611-625): d = Rlc (s g) + tlc - q,
//     dd_i = sum_j g_j W_ij + s.v (Rlc.a g)_i + tlc_i.v,   W_ij = s.a Rlc_ij.v   (candidate table, lin_table)
//   3-D/2-D (IBA_PlaneFactor, IBACalib2.hpp:152-184): the keypoint ray C = (Cxz, Cyz, 1) is constant, P0 = Z0 C,
//     dZ0 = (dnum - Z0 dden) / den with dp0c = R.v p0 + t.v, dn0c = R.v n0  (folded into 12 scalar weights of R.v and t.v);
//     row s: dP1 = (rp C) dZ0 + rp_3 ds, so deu = alpha dZ0 + beta ds (and dev likewise): two scalars per row.
#pragma once
#include "dual.cuh"

namespace stl {

// a residual and its seven partials
struct Row7 {
    double a;
    double v[7];
};

// W[3i+j][k] = s.a * Rlc_ij.v[k]
STL_HD void lin_table(const LmCand &c, double (*W)[7], int first, int step) {
    for (int m = first; m < 63; m += step) W[m / 7][m % 7] = c.s.a * c.Rlc[m / 7].v[m % 7];
}

// ---- 3-D/3-D: g = map point (3), scan point q (3), normal n (3)
// the three values of d, as the dual evaluation forms them (Ms = s*g, mv3(Rlc, Ms), + tlc, - q)
STL_HD void p3_values(const LmCand &c, const double *g, double *d) {
    const double m0 = c.s.a * g[0], m1 = c.s.a * g[1], m2 = c.s.a * g[2];
    for (int i = 0; i < 3; ++i) d[i] = (((c.Rlc[i * 3].a * m0 + c.Rlc[i * 3 + 1].a * m1) + c.Rlc[i * 3 + 2].a * m2) + c.tlc[i].a) - g[3 + i];
}
// partials of d_i, times w, added to v
STL_HD void p3_partials(const LmCand &c, const double (*W)[7], const double *g, int i, double w, double *v) {
    const double rg = fma(c.Rlc[i * 3 + 2].a, g[2], fma(c.Rlc[i * 3 + 1].a, g[1], c.Rlc[i * 3].a * g[0]));
#pragma unroll
    for (int k = 0; k < 7; ++k) {
        const double dk = fma(g[2], W[i * 3 + 2][k], fma(g[1], W[i * 3 + 1][k], fma(g[0], W[i * 3][k], fma(c.s.v[k], rg, c.tlc[i].v[k]))));
        v[k] = fma(w, dk, v[k]);
    }
}
// point-to-point row i
STL_HD Row7 p3_point_row(const LmCand &c, const double (*W)[7], const double *g, const double *d, int i) {
    Row7 r;
    r.a = d[i];
    for (int k = 0; k < 7; ++k) r.v[k] = 0.0;
    p3_partials(c, W, g, i, 1.0, r.v);
    return r;
}
// point-to-plane row: e = d . n
STL_HD Row7 p3_plane_row(const LmCand &c, const double (*W)[7], const double *g, const double *d) {
    Row7 r;
    r.a = (d[0] * g[6] + d[1] * g[7]) + d[2] * g[8];
    for (int k = 0; k < 7; ++k) r.v[k] = 0.0;
    for (int i = 0; i < 3; ++i) p3_partials(c, W, g, i, g[6 + i], r.v);
    return r;
}

// ---- 3-D/2-D: g = plane point p0 (3), normal n0 (3) in the keyframe's camera at the LiDAR frame; C = (Cxz, Cyz, 1)
// depth Z0 of the keypoint ray on the plane (value as the dual division forms it) and its partials
STL_HD void p2_depth(const LmCand &c, const double *g, double Cxz, double Cyz, double &Z0, double *dZ) {
    double p0c[3], n0c[3];
    for (int i = 0; i < 3; ++i) {
        p0c[i] = ((c.R[i * 3].a * g[0] + c.R[i * 3 + 1].a * g[1]) + c.R[i * 3 + 2].a * g[2]) + c.t[i].a;
        n0c[i] = (c.R[i * 3].a * g[3] + c.R[i * 3 + 1].a * g[4]) + c.R[i * 3 + 2].a * g[5];
    }
    const double num = (n0c[0] * p0c[0] + n0c[1] * p0c[1]) + n0c[2] * p0c[2];
    const double den = (n0c[0] * Cxz + n0c[1] * Cyz) + n0c[2];
    const double gi = 1.0 / den;
    Z0 = num * gi;
    // dnum - Z0 dden = sum_ij R_ij.v (n0c_i p0_j + (p0c_i - Z0 C_i) n0_j) + sum_i n0c_i t_i.v
    const double Cz[3] = {Cxz, Cyz, 1.0};
    double H[9];
    for (int i = 0; i < 3; ++i) {
        const double e = fma(-Z0, Cz[i], p0c[i]);
        for (int j = 0; j < 3; ++j) H[i * 3 + j] = fma(e, g[3 + j], n0c[i] * g[j]);
    }
#pragma unroll
    for (int k = 0; k < 7; ++k) {
        double x = fma(n0c[2], c.t[2].v[k], fma(n0c[1], c.t[1].v[k], n0c[0] * c.t[0].v[k]));
#pragma unroll
        for (int m = 0; m < 9; ++m) x = fma(H[m], c.R[m].v[k], x);
        dZ[k] = x * gi;
    }
}
// P1 = rp (Z0 C) + rp_3 s for one covisible keyframe (rp: its 3x4 relative pose), values as both passes form them
STL_HD void p2_point(const LmCand &c, const float *rp, double Z0, double Cxz, double Cyz, double *P1) {
    const double P0[3] = {Z0 * Cxz, Z0 * Cyz, Z0};
    for (int i = 0; i < 3; ++i)
        P1[i] = (((double)rp[i * 4] * P0[0] + (double)rp[i * 4 + 1] * P0[1]) + (double)rp[i * 4 + 2] * P0[2]) + (double)rp[i * 4 + 3] * c.s.a;
}
// the reprojection rows (eu, ev) of one covisible keyframe: values as the dual evaluation forms them ((P1_0 fx) / P1_2 with the
// dual division's reciprocal), partials alpha dZ0 + beta ds
STL_HD void p2_rows(const LmCand &c, const float *rp, const double *P1, const double *dZ, double Cxz, double Cyz, double fx, double fy,
                    double cx, double cy, float u, float v, Row7 &eu, Row7 &ev) {
    const double gi = 1.0 / P1[2];
    const double qu = (P1[0] * fx) * gi, qv = (P1[1] * fy) * gi;
    eu.a = (qu + cx) - (double)u;
    ev.a = (qv + cy) - (double)v;
    double a[3], b[3];  // dP1_i = a_i dZ0 + b_i ds
    for (int i = 0; i < 3; ++i) {
        a[i] = fma((double)rp[i * 4 + 1], Cyz, (double)rp[i * 4] * Cxz) + (double)rp[i * 4 + 2];
        b[i] = (double)rp[i * 4 + 3];
    }
    const double au = fma(-qu, a[2], fx * a[0]) * gi, bu = fma(-qu, b[2], fx * b[0]) * gi;
    const double av = fma(-qv, a[2], fy * a[1]) * gi, bv = fma(-qv, b[2], fy * b[1]) * gi;
#pragma unroll
    for (int k = 0; k < 7; ++k) {
        eu.v[k] = fma(au, dZ[k], bu * c.s.v[k]);
        ev.v[k] = fma(av, dZ[k], bv * c.s.v[k]);
    }
}

}  // namespace stl
