"""The oversize-keyframe adapters without a GPU: stl::Context::allow_oversize_keyframes / oversize_keyframes
(include/stlcalib_host.hpp) compile and follow the count-then-fill protocol of stl_oversize_keyframes against a stub of the
C-ABI, and the Python wrappers validate their arguments before they reach the library."""
import ctypes as C
import importlib
import os
import subprocess

import numpy as np
import pytest

from conftest import PKG

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SRC = r"""
#include <cstdio>
#include "stlcalib_host.hpp"
static int32_t g_allow = -1;
static stl_ctx_t *const g_ctx = reinterpret_cast<stl_ctx_t *>(0x10);
static const int32_t g_ov[3] = {2, 5, 9};
extern "C" {
stl_status_t stl_create(const stl_params_t *, int32_t, stl_ctx_t **out) { *out = g_ctx; return STL_OK; }
void stl_destroy(stl_ctx_t *) {}
const char *stl_last_error(const stl_ctx_t *) { return ""; }
stl_status_t stl_allow_oversize_keyframes(stl_ctx_t *, int32_t allow) { g_allow = allow; return STL_OK; }
stl_status_t stl_oversize_keyframes(stl_ctx_t *, int32_t *kf, int32_t cap, int32_t *n) {
    *n = 3;
    for (int i = 0; i < cap && i < 3; ++i) if (kf) kf[i] = g_ov[i];
    return STL_OK;
}
}
int main() {
    stl_params_t p{};
    stl::Context ctx(p);
    int bad = 0;
    ctx.allow_oversize_keyframes(true);
    bad |= (g_allow != 1) << 0;
    ctx.allow_oversize_keyframes(false);
    bad |= (g_allow != 0) << 1;
    const std::vector<int32_t> kf = ctx.oversize_keyframes();
    bad |= (kf != std::vector<int32_t>{2, 5, 9}) << 2;
    std::printf("%d\n", bad);
    return bad;
}
"""


def test_oversize_adapter_compiles_and_fills(tmp_path):
    src, exe = tmp_path / "oversize_stub.cpp", tmp_path / "oversize_stub"
    src.write_text(SRC)
    r = subprocess.run(["/usr/bin/g++", "-std=c++17", "-Wall", "-O1", "-I" + os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, f"failed checks (bit mask): {r.stdout}"


class _FakeLib:
    """Records the C-ABI calls of the wrappers; stl_oversize_keyframes reports keyframes 1 and 4."""

    def __init__(self):
        self.calls = []

    def stl_allow_oversize_keyframes(self, h, allow):
        self.calls.append(("allow", allow))
        return 0

    def stl_oversize_keyframes(self, h, kf, cap, n):
        n._obj.value = 2
        if kf and cap >= 2:
            C.cast(kf, C.POINTER(C.c_int32))[0] = 1
            C.cast(kf, C.POINTER(C.c_int32))[1] = 4
        return 0


def _ctx():
    capi = importlib.import_module(PKG + ".capi")
    c = capi.Context.__new__(capi.Context)  # no device: only the argument handling runs
    c.lib, c.h = _FakeLib(), None
    return c


@pytest.mark.parametrize("flag", [True, False, 1, 0, np.bool_(True)])
def test_allow_oversize_accepts_bools(flag):
    c = _ctx()
    c.allow_oversize_keyframes(flag)
    assert c.lib.calls == [("allow", 1 if flag else 0)]


@pytest.mark.parametrize("flag", [2, -1, "yes", None, 1.0])
def test_allow_oversize_rejects_other_values(flag):
    c = _ctx()
    with pytest.raises(TypeError):
        c.allow_oversize_keyframes(flag)
    assert c.lib.calls == []


def test_oversize_keyframes_returns_int32_list():
    got = _ctx().oversize_keyframes()
    assert got.dtype == np.int32 and got.tolist() == [1, 4]


def test_oversize_symbols_are_bound():
    abi = importlib.import_module(PKG + "._abi")
    assert {"stl_allow_oversize_keyframes", "stl_oversize_keyframes"} <= set(abi.CALIB_SYMBOLS)
