"""Deterministic stand-ins for the optimisers the reference links against (NOMAD 4 and Ceres are
not vendored and are absent from this image).  They exist so that the end-to-end statement of the
parity bar — *the final extrinsic after the unchanged optimiser agrees to 0.01 deg / 0.1 cm* — can be
tested: the same driver runs once over the GPU evaluator and once over the CPU oracle.

They are NOT a replacement for NOMAD / Ceres; INTEGRATION.md shows how the real ones bind.

* :func:`poll_search`  — the shape of the NOMAD run in ``iba_global.cpp:551-599``: bounded variables,
  objective + three progressive-barrier constraints (``BB_OUTPUT_TYPE OBJ PB PB PB``), an evaluation
  budget (``MAX_BB_EVAL``), an initial frame size and a minimum mesh size.  Each iteration polls the
  2N coordinate directions (``DIRECTION_TYPE ORTHO 2N``) and hands the whole poll set to
  ``evaluator.eval_block`` — one device call per iteration.
* :func:`lm_refine`    — the shape of ``iba_local.cpp:434-460``: outer loop = ``BuildProblem`` at the
  current estimate (association), inner loop = Levenberg-Marquardt on the frozen residual blocks,
  stop when the estimate moved less than ``iba_min_diff``.
* :func:`lm_refine_multi` — :func:`lm_refine` from several starts in lockstep over a problem set: one
  ``evaluate`` call per inner iteration for all starts still iterating, one ``build`` per outer iteration
  for the starts not yet converged.  Start p follows exactly the trajectory of ``lm_refine`` from ``X0[p]``.
"""
from __future__ import annotations

import numpy as np


def _violation(bbo) -> float:
    """Progressive-barrier aggregate h(x) = sum max(c_j, 0)^2 over the PB outputs."""
    c = np.asarray(bbo[1:], dtype=np.float64)
    if np.isnan(c).any():
        return float("inf")
    return float((np.maximum(c, 0.0) ** 2).sum())


def _better(fa, ha, fb, hb) -> bool:
    """(f, h) of a dominates b: feasible beats infeasible, then smaller h, then smaller f."""
    if ha == 0.0 and hb == 0.0:
        return fa < fb
    if ha != hb:
        return ha < hb
    return fa < fb


def poll_search(evaluator, x0, lb, ub, max_bb_eval=200, init_frame=None, min_mesh=1e-6):
    """Coordinate poll with frame halving.  ``evaluator.eval_block(X)`` returns rows ``[f, C1, C2, C3]``.

    Returns ``(x_best, bbo_best, n_eval, history)``; fully deterministic for a deterministic evaluator."""
    x = np.asarray(x0, dtype=np.float64).copy()
    lb = np.asarray(lb, dtype=np.float64)
    ub = np.asarray(ub, dtype=np.float64)
    n = x.size
    frame = np.asarray(init_frame if init_frame is not None else 0.1 * (ub - lb), dtype=np.float64).copy()
    bbo = np.asarray(evaluator.eval_block(x[None])[0], dtype=np.float64)
    f, h = float(bbo[0]), _violation(bbo)
    n_eval = 1
    history = [(n_eval, f, h)]
    while n_eval + 2 * n <= max_bb_eval and frame.max() > min_mesh:
        P = np.repeat(x[None], 2 * n, axis=0)
        for i in range(n):
            P[2 * i, i] = min(x[i] + frame[i], ub[i])
            P[2 * i + 1, i] = max(x[i] - frame[i], lb[i])
        out = np.asarray(evaluator.eval_block(P), dtype=np.float64)
        n_eval += 2 * n
        best = -1
        bf, bh = f, h
        for j in range(2 * n):  # fixed scan order: ties keep the first
            fj, hj = float(out[j, 0]), _violation(out[j])
            if np.isfinite(fj) and _better(fj, hj, bf, bh):
                best, bf, bh = j, fj, hj
        if best >= 0:
            x, bbo, f, h = P[best].copy(), out[best].copy(), bf, bh
        else:
            frame *= 0.5
        history.append((n_eval, f, h))
    return x, bbo, n_eval, history


def lm_refine(problem, x0, max_iba_iter=5, max_num_iterations=30, iba_min_diff=1e-6, lam0=1e-4):
    """``problem.build(x)`` freezes the residual blocks at x (BuildProblem); ``problem.evaluate(x)`` returns
    ``(cost, g[7], H[7,7])`` of those blocks (what Ceres assembles).  Returns ``(x, costs)``."""
    x = np.asarray(x0, dtype=np.float64).copy()
    costs = []
    for _ in range(max_iba_iter):
        last = x.copy()
        problem.build(x)
        lam = lam0
        cost, g, H = problem.evaluate(x)
        for _ in range(max_num_iterations):
            D = np.diag(np.maximum(np.diag(H), 1e-12))
            try:
                step = -np.linalg.solve(H + lam * D, g)
            except np.linalg.LinAlgError:
                lam *= 10.0
                continue
            c1, g1, H1 = problem.evaluate(x + step)
            if np.isfinite(c1) and c1 < cost:
                x = x + step
                rel = (cost - c1) / max(cost, 1e-300)
                cost, g, H = c1, g1, H1
                lam = max(lam / 3.0, 1e-12)
                if rel < 1e-10:
                    break
            else:
                lam *= 4.0
                if lam > 1e8:
                    break
        costs.append(cost)
        if np.allclose(last, x, rtol=0.0, atol=iba_min_diff):  # allClose(last_sim3_log, sim3_log, iba_min_diff)
            break
    return x, costs


def lm_refine_multi(problem_set, X0, max_iba_iter=5, max_num_iterations=30, iba_min_diff=1e-6, lam0=1e-4):
    """:func:`lm_refine` for P starts at once.  ``problem_set.build(X, rebuild)`` freezes problem p at X[p] for the starts
    flagged in ``rebuild`` (None: a new set of P); ``problem_set.evaluate(X, problem)`` returns ``(cost [B], g [B,7],
    H [B,7,7])`` of row b of X on problem ``problem[b]``.  Returns ``(X [P,7], costs per start)``."""
    X = np.array(np.atleast_2d(X0), dtype=np.float64)
    P = X.shape[0]
    costs = [[] for _ in range(P)]
    outer = np.ones(P, dtype=bool)  # starts whose outer loop goes on
    for it in range(max_iba_iter):
        act = np.flatnonzero(outer)
        if act.size == 0:
            break
        last = X.copy()
        problem_set.build(X, None if it == 0 else outer.astype(np.uint8))
        lam = np.full(P, lam0)
        cost, g, H = np.zeros(P), np.zeros((P, 7)), np.zeros((P, 7, 7))
        c, gg, HH = problem_set.evaluate(X[act], act)
        cost[act], g[act], H[act] = c, gg, HH
        inner = outer.copy()  # starts whose inner loop goes on
        for _ in range(max_num_iterations):
            todo, steps = [], []
            for p in np.flatnonzero(inner):
                D = np.diag(np.maximum(np.diag(H[p]), 1e-12))
                try:
                    step = -np.linalg.solve(H[p] + lam[p] * D, g[p])
                except np.linalg.LinAlgError:
                    lam[p] *= 10.0
                    continue
                todo.append(p)
                steps.append(step)
            if not todo:
                if not inner.any():
                    break
                continue
            todo = np.asarray(todo)
            Xt = X[todo] + np.asarray(steps)
            c1, g1, H1 = problem_set.evaluate(Xt, todo)
            for k, p in enumerate(todo):
                if np.isfinite(c1[k]) and c1[k] < cost[p]:
                    X[p] = Xt[k]
                    rel = (cost[p] - c1[k]) / max(cost[p], 1e-300)
                    cost[p], g[p], H[p] = c1[k], g1[k], H1[k]
                    lam[p] = max(lam[p] / 3.0, 1e-12)
                    if rel < 1e-10:
                        inner[p] = False
                else:
                    lam[p] *= 4.0
                    if lam[p] > 1e8:
                        inner[p] = False
            if not inner.any():
                break
        for p in act:
            costs[p].append(cost[p])
            if np.allclose(last[p], X[p], rtol=0.0, atol=iba_min_diff):
                outer[p] = False
    return X, costs
