"""Host-side mirror of the reference's call signatures for the cost-evaluation path.

The reference is C++; its C++-side adapters live in include/stlcalib_host.hpp.  This module
mirrors the same interface for Python callers and for the parity tests, on top of the C-ABI:

* :func:`BAError`            <- ``BAError(xvec, PointClouds, KdTrees, vTwl, KFIdMap, KeyFrames,
                                 iba_params, multiprocessing, verborse)`` (iba_global.cpp:169-173,
                                 iba_func.cpp:179-183): returns (f1, f2, C, valid_cnt_3d_2d, cnt_3d_2d)
* :class:`BALoss`            <- ``class BALoss : NOMAD::Evaluator`` (iba_global.cpp:346-405):
                                 ``eval_x`` -> the BBO values "f C1 C2 C3"; ``eval_block`` for a poll batch
* :func:`evaluate_sim3_list` <- the iba_func main loop (iba_func.cpp:458-470): one row
                                 ``f1 f2 C valid_rate`` per candidate
* :class:`LMProblem`         <- BuildProblem + ceres::Problem::Evaluate (iba_local.cpp:145-323,434-446):
                                 associate at the current estimate, then cost / J^T r / J^T J
* :class:`LMProblemSet`      <- the same for several starts at once: one ceres::Problem per start,
                                 all frozen on one context and evaluated by one call

All state (scans, keyframes, index) lives in a :class:`capi.Context`; with several GPUs the
keyframes are sharded (parallel.py) and the partial sums all-reduced before the epilogue.
"""
from __future__ import annotations

import numpy as np

from . import _abi
from .capi import Context


def BAError(xvec, ctx: Context, allreduce=None, verborse: bool = False):
    """One candidate -> (f1, f2, C, valid_cnt_3d_2d, cnt_3d_2d), exactly BAError's return tuple.

    ``allreduce`` (optional) sums the [1,12] partial-sum row over keyframe shards."""
    sums = ctx.eval_sums(np.asarray(xvec, dtype=np.float64).reshape(1, 7))
    if allreduce is not None:
        sums = allreduce(sums)
    out = ctx.finalize(sums[0])
    if verborse:  # iba_global.cpp:341-342
        print("plane: %d, point: %d 3d-2d: %d" % (int(sums[0, 8]), int(sums[0, 9]), int(sums[0, 5])))
    return out


class BALoss:
    """Nomad evaluator shape (iba_global.cpp:346-405): same inputs (7 doubles), same outputs
    (BBO = f, C1, C2, C3), ``countEval = True``, returns True."""

    def __init__(self, ctx: Context, allreduce=None):
        self.ctx = ctx
        self.allreduce = allreduce

    def eval_x(self, x):
        ba = BAError(x, self.ctx, self.allreduce)
        bbo = self.ctx.bbo(ba)
        return True, True, bbo  # (return value, countEval, BBO)

    def bbo_string(self, x) -> str:
        """The string handed to ``x.setBBO`` (iba_global.cpp:389-393)."""
        _, _, bbo = self.eval_x(x)
        return " ".join(repr(float(v)) for v in bbo)

    def eval_block(self, X):
        """A whole poll batch in one device call (Nomad 4 ``eval_block``)."""
        X = np.ascontiguousarray(np.atleast_2d(X), dtype=np.float64)
        sums = self.ctx.eval_sums(X)
        if self.allreduce is not None:
            sums = self.allreduce(sums)
        return [self.ctx.bbo(self.ctx.finalize(r)) for r in sums]


def evaluate_sim3_list(ctx: Context, X, allreduce=None) -> np.ndarray:
    """iba_func (iba_func.cpp:458-470): rows of ``f1 f2 C valid_rate`` for a list of Sim3 logs."""
    X = np.ascontiguousarray(np.atleast_2d(X), dtype=np.float64)
    sums = ctx.eval_sums(X)
    if allreduce is not None:
        sums = allreduce(sums)
    rows = []
    for r in sums:
        f1, f2, C, valid, cnt = ctx.finalize(r)
        rows.append((f1, f2, C, valid / cnt if cnt else float("nan")))  # iba_func.cpp:466
    return np.asarray(rows)


class LMProblem:
    """ceres::Problem over one 7-double block, frozen by BuildProblem (iba_local.cpp:443)."""

    def __init__(self, ctx: Context, allreduce=None):
        self.ctx = ctx
        self.allreduce = allreduce
        self.n_blocks = None

    def build(self, x0):
        self.n_blocks = self.ctx.associate(x0)
        return self.n_blocks

    def evaluate(self, x):
        """-> (cost, gradient[7], JtJ[7,7]) at x (ceres::Problem::Evaluate with Huber applied)."""
        s = self.ctx.linearize(np.asarray(x, dtype=np.float64).reshape(1, 7))
        if self.allreduce is not None:
            s = self.allreduce(s)
        return float(s[0, 0]), s[0, 1:8].copy(), s[0, 8:57].reshape(7, 7).copy()

    def blocks(self, x):
        """The residual blocks one by one (raw residuals + Jacobian rows, no robust kernel): what
        ceres::CostFunction::Evaluate / g2o computeError + linearizeOplus return per block."""
        return self.ctx.eval_blocks(x)

    def lm_step(self, x, lam: float):
        """One damped Gauss-Newton step on the raw 7 parameters (VertexSim3 oplus is '+')."""
        cost, g, H = self.evaluate(x)
        A = H + lam * np.diag(np.maximum(np.diag(H), 1e-12))
        dx = -np.linalg.solve(A, g)
        return np.asarray(x) + dx, cost


class LMProblemSet:
    """P independent :class:`LMProblem` s on one context (multi-start refinement): problem p is frozen at its own start."""

    def __init__(self, ctx: Context, allreduce=None):
        self.ctx = ctx
        self.allreduce = allreduce
        self.n_blocks = None

    def build(self, X0, rebuild=None):
        """BuildProblem at X0[p] for every start ([P,7]); rebuild (mask [P]) re-associates only the flagged problems."""
        self.n_blocks = self.ctx.associate_multi(X0, rebuild)
        return self.n_blocks

    def evaluate(self, X, problem=None):
        """-> (cost [B], gradient [B,7], JtJ [B,7,7]) of candidate b (X [B,7]) on problem problem[b] (None: candidate p on problem p)."""
        s = self.ctx.linearize_multi(np.atleast_2d(np.asarray(X, dtype=np.float64)), problem)
        if self.allreduce is not None:
            s = self.allreduce(s)
        return s[:, 0].copy(), s[:, 1:8].copy(), s[:, 8:57].reshape(-1, 7, 7).copy()


# ------------------------------------------------------------------------------------------------
# N4 — the steps before the cost evaluation, on the same 7 parameters
class HandEyeInit:
    """``HECalibRobustKernelg2o`` / ``HECalibLineProcessg2o`` (include/NLHECalib.hpp:118-278) with the edges evaluated
    through an evaluator ``lin(edges, x) -> ([B,62], chi2 [B,n])`` — :meth:`capi.Context.he_linearize` on the GPU or the
    oracle on the CPU.  The g2o optimiser itself (Dogleg / Levenberg with ``optimize(10)``) is third-party and not
    available here: a damped Gauss-Newton loop on the returned (g, H) stands in for it, identically for both
    evaluators, so the two final extrinsics can be compared."""

    def __init__(self, lin):
        self.lin = lin

    def _solve(self, edges, x, iters=10):
        lam = 1e-4
        L, _ = self.lin(edges, x[None])
        cost, g, H = L[0, 0], L[0, 1:8], L[0, 8:57].reshape(7, 7)
        for _ in range(iters):
            step = -np.linalg.solve(H + lam * np.diag(np.maximum(np.diag(H), 1e-12)), g)
            L1, _ = self.lin(edges, (x + step)[None])
            if L1[0, 0] < cost:
                x = x + step
                cost, g, H = L1[0, 0], L1[0, 1:8], L1[0, 8:57].reshape(7, 7)
                lam = max(lam / 3.0, 1e-12)
            else:
                lam *= 4.0
        return x, cost

    def robust_kernel(self, edges, x0, iters=10):
        """Huber kernel on every motion edge + the regularisation edge (NLHECalib.hpp:118-158)."""
        return self._solve(edges, np.asarray(x0, dtype=np.float64).copy(), iters)

    def line_process(self, edges, x0, mu0=64.0, divid_factor=1.4, min_mu=1e-1, ex_max_iter=20, regulation_ratio=0.005):
        """Graduated re-weighting w = mu / (mu + chi2), information = w^2 I (NLHECalib.hpp:224-246)."""
        import copy
        ed = copy.copy(edges)
        ed.huber_delta = 0.0
        ed.info = None
        x, cost = self._solve(ed, np.asarray(x0, dtype=np.float64).copy())
        mu = mu0
        for _ in range(ex_max_iter):
            ed.info = None
            _, chi2 = self.lin(ed, x[None])       # chi2 with identity information
            w2 = (mu / (mu + chi2[0])) ** 2
            ed.info = np.ascontiguousarray(w2)
            if edges.regulation > 0:
                ed.regulation = float(w2.sum() * regulation_ratio)
            x, cost = self._solve(ed, x)
            mu /= divid_factor
            if mu < min_mu:
                break
        return x, cost


def calib_ba(lin, edges, x0, rounds=4, iters=10, chi2_max=5.991):
    """``Optimizer::OptimizeExtrinsicGlobal`` (Optimizer.cc:1583-1744): four rounds of ten iterations from the SAME start,
    edges re-classified as outliers (level 1) by chi2 > 5.991 after every round, the robust kernel dropped after the
    third.  ``lin(edges, x) -> ([B,62], chi2)``.  Returns (x, inliers)."""
    import copy
    ed = copy.copy(edges)
    ed.level = np.zeros(edges.n_edges, np.uint8)
    x0 = np.asarray(x0, dtype=np.float64)
    x = x0.copy()
    he = HandEyeInit(lin)
    for it in range(rounds):
        x, _ = he._solve(ed, x0.copy(), iters)       # v->setEstimate(p_tcl) at the start of every round
        _, chi2 = lin(ed, x[None])
        ed.level = (chi2[0] > chi2_max).astype(np.uint8)
        if it == 2:
            ed.huber_delta = 0.0                        # e->setRobustKernel(0)
    return x, int((ed.level == 0).sum())
