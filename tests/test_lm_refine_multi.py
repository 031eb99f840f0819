"""lm_refine_multi over a numpy problem set: every start follows lm_refine's trajectory exactly, and the rebuild masks
re-associate only the starts whose outer loop is still running (no GPU)."""
import importlib

import numpy as np

optim = importlib.import_module("spatial-temporal-lidar-camera-calibration_b200.optim")

_RNG = np.random.default_rng(7)
_A = _RNG.normal(size=(40, 7))
_B = _RNG.normal(size=40)


def _frozen(x0):
    """'Association' at x0: the residuals whose value at x0 is small enough are kept (a kink in the cost as x0 moves)."""
    r = _A @ x0 - _B
    return np.abs(r) < 2.5


def _lin(x, keep, delta=0.7):
    """Huber cost, gradient and Gauss-Newton H of the kept residuals (Ceres' Corrector scaling)."""
    r = (_A @ x - _B)[keep]
    J = _A[keep]
    a = np.abs(r)
    rho = np.where(a > delta, 2 * delta * a - delta * delta, r * r)
    sr = np.where(a > delta, np.sqrt(delta / np.maximum(a, 1e-300)), 1.0)
    rs, Js = sr * r, sr[:, None] * J
    return 0.5 * rho.sum(), Js.T @ rs, Js.T @ Js


class _One:
    def __init__(self):
        self.keep = None

    def build(self, x):
        self.keep = _frozen(np.asarray(x))

    def evaluate(self, x):
        return _lin(np.asarray(x), self.keep)


class _Set:
    def __init__(self):
        self.keep = None
        self.masks = []

    def build(self, X, rebuild=None):
        X = np.atleast_2d(X)
        if rebuild is None:
            self.keep = [_frozen(x) for x in X]
            self.masks.append(None)
        else:
            assert len(rebuild) == len(self.keep)
            self.masks.append(np.asarray(rebuild, bool).copy())
            for p in np.flatnonzero(rebuild):
                self.keep[p] = _frozen(X[p])

    def evaluate(self, X, problem=None):
        X = np.atleast_2d(X)
        problem = np.arange(len(X)) if problem is None else np.asarray(problem)
        out = [_lin(x, self.keep[p]) for x, p in zip(X, problem)]
        return np.array([o[0] for o in out]), np.array([o[1] for o in out]), np.array([o[2] for o in out])


def test_multi_equals_single_per_start():
    X0 = _RNG.normal(scale=0.8, size=(6, 7))
    X0[0] = optim.lm_refine(_One(), X0[1], max_iba_iter=10, iba_min_diff=1e-12)[0]  # a start at a fixed point: one outer iteration
    kw = dict(max_iba_iter=8, max_num_iterations=25, iba_min_diff=1e-6)
    S = _Set()
    X, costs = optim.lm_refine_multi(S, X0, **kw)
    n_outer = []
    for p in range(len(X0)):
        x1, c1 = optim.lm_refine(_One(), X0[p], **kw)
        assert np.array_equal(X[p], x1), p
        assert costs[p] == c1, p
        n_outer.append(len(c1))
    assert len(set(n_outer)) > 1, "the starts should converge after different numbers of outer iterations"
    # the first build makes the set; every later one re-associates exactly the starts whose outer loop is still running
    assert S.masks[0] is None
    for k, m in enumerate(S.masks[1:], start=1):
        assert np.array_equal(m, np.array([n > k for n in n_outer])), k
    assert len(S.masks) == max(n_outer)


def test_single_start():
    x0 = _RNG.normal(scale=0.5, size=7)
    X, costs = optim.lm_refine_multi(_Set(), x0[None])
    x1, c1 = optim.lm_refine(_One(), x0)
    assert np.array_equal(X[0], x1) and costs[0] == c1
