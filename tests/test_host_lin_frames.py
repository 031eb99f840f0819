"""The per-keyframe linearisation adapters without a GPU: stl::Context::linearize_frames (include/stlcalib_host.hpp) sizes its
buffer B x n_kf rows and hands the problem pointer through to stl_linearize_frames (built and run against a stub of the C-ABI),
and Context.linearize_frames checks the shapes of X and problem before it reaches the library."""
import ctypes as C
import importlib
import os
import subprocess
from types import SimpleNamespace

import numpy as np
import pytest

from conftest import PKG

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SRC = r"""
#include <cstdio>
#include "stlcalib_host.hpp"
static stl_ctx_t *const g_ctx = reinterpret_cast<stl_ctx_t *>(0x10);
static const double *g_x = nullptr;
static int32_t g_B = -1;
static const int32_t *g_problem = reinterpret_cast<const int32_t *>(0x1);
extern "C" {
stl_status_t stl_create(const stl_params_t *, int32_t, stl_ctx_t **out) { *out = g_ctx; return STL_OK; }
void stl_destroy(stl_ctx_t *) {}
const char *stl_last_error(const stl_ctx_t *) { return ""; }
stl_status_t stl_linearize_frames(stl_ctx_t *ctx, const double *x, int32_t B, const int32_t *problem, stl_lin_sums_t *out) {
    g_x = x; g_B = B; g_problem = problem;
    for (int r = 0; r < B * 3; ++r) { out[r].cost = r; out[r].n_residuals = 10 * r; }  // every row of a [B][3] buffer
    return ctx == g_ctx ? STL_OK : STL_ERR_INVALID;
}
}
int main() {
    stl_params_t p{};
    stl::Context ctx(p);
    int bad = 0;
    const double x[2 * 7] = {0};
    const int32_t prob[2] = {1, 0};
    std::vector<stl_lin_sums_t> r = ctx.linearize_frames(x, 2, 3, prob);
    bad |= (r.size() != 6) << 0;
    bad |= (g_x != x || g_B != 2 || g_problem != prob) << 1;
    for (int i = 0; i < (int)r.size(); ++i) bad |= (r[i].cost != i || r[i].n_residuals != 10 * i) << 2;
    r = ctx.linearize_frames(x, 2, 3);
    bad |= (g_problem != nullptr || r.size() != 6) << 3;
    std::printf("%d\n", bad);
    return bad;
}
"""


def test_linearize_frames_adapter_sizes_rows_and_passes_problem(tmp_path):
    src, exe = tmp_path / "lin_frames_stub.cpp", tmp_path / "lin_frames_stub"
    src.write_text(SRC)
    r = subprocess.run(["/usr/bin/g++", "-std=c++17", "-Wall", "-O1", "-I" + os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, f"failed checks (bit mask): {r.stdout}"


class _FakeLib:
    """Records stl_linearize_frames calls and fills every row with its flat index."""

    def __init__(self):
        self.calls = []

    def stl_linearize_frames(self, h, x, B, problem, out):
        p = None if problem is None else [C.cast(problem, C.POINTER(C.c_int32))[i] for i in range(B)]
        self.calls.append((B, p))
        return 0


def _ctx(n_kf=5):
    capi = importlib.import_module(PKG + ".capi")
    c = capi.Context.__new__(capi.Context)  # no device: only the argument handling runs
    c.lib, c.h = _FakeLib(), None
    c.pack = SimpleNamespace(n_kf=n_kf)
    return c


def test_linearize_frames_shape_and_problem_passthrough():
    c = _ctx(5)
    out = c.linearize_frames(np.zeros((3, 7)), problem=[2, 0, 1])
    assert out.shape == (3, 5, 62) and out.dtype == np.float64
    out = c.linearize_frames(np.zeros(7))  # one candidate as a flat vector
    assert out.shape == (1, 5, 62)
    assert c.lib.calls == [(3, [2, 0, 1]), (1, None)]


@pytest.mark.parametrize("X", [np.zeros((2, 6)), np.zeros((2, 8)), np.zeros((2, 7, 1)), np.zeros((0, 7)), np.zeros(5)])
def test_linearize_frames_rejects_bad_x(X):
    c = _ctx()
    with pytest.raises(ValueError):
        c.linearize_frames(X)
    assert c.lib.calls == []


@pytest.mark.parametrize("problem", [[0], [0, 1, 2], np.zeros((3, 1), np.int32)])
def test_linearize_frames_rejects_problem_of_other_length(problem):
    c = _ctx()
    with pytest.raises(ValueError):
        c.linearize_frames(np.zeros((2, 7)), problem=problem)
    assert c.lib.calls == []


def test_linearize_frames_symbol_is_bound():
    abi = importlib.import_module(PKG + "._abi")
    assert "stl_linearize_frames" in abi.CALIB_SYMBOLS
