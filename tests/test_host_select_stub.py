"""stl::Context::select_keyframes / select_all (include/stlcalib_host.hpp) hand the C-ABI the pointer that means what they
say: an empty list selects NO keyframe, so it must arrive as a non-null pointer with n = 0 (NULL means every keyframe), whatever
the vector's history; select_all passes NULL.  Built and run against a stub of the C-ABI (no GPU, no library)."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SRC = r"""
#include <cstdio>
#include "stlcalib_host.hpp"
static const int32_t *g_kf = nullptr;
static int32_t g_n = -1;
static stl_ctx_t *const g_ctx = reinterpret_cast<stl_ctx_t *>(0x10);
extern "C" {
stl_status_t stl_create(const stl_params_t *, int32_t, stl_ctx_t **out) { *out = g_ctx; return STL_OK; }
void stl_destroy(stl_ctx_t *) {}
const char *stl_last_error(const stl_ctx_t *) { return ""; }
stl_status_t stl_select_keyframes(stl_ctx_t *, const int32_t *kf, int32_t n) { g_kf = kf; g_n = n; return STL_OK; }
}
int main() {
    stl_params_t p{};
    stl::Context ctx(p);
    int bad = 0;
    ctx.select_keyframes({});                                   // a fresh empty vector (data() may be null)
    bad |= (g_kf == nullptr || g_n != 0) << 0;
    std::vector<int32_t> v;
    ctx.select_keyframes(v);
    bad |= (g_kf == nullptr || g_n != 0) << 1;
    v = {1, 4};
    ctx.select_keyframes(v);
    bad |= (g_kf != v.data() || g_n != 2) << 2;
    v.clear();                                                  // emptied after an allocation
    ctx.select_keyframes(v);
    bad |= (g_kf == nullptr || g_n != 0) << 3;
    ctx.select_all();
    bad |= (g_kf != nullptr || g_n != 0) << 4;
    std::printf("%d\n", bad);
    return bad;
}
"""


def test_select_adapter_passes_empty_lists_as_non_null(tmp_path):
    src, exe = tmp_path / "select_stub.cpp", tmp_path / "select_stub"
    src.write_text(SRC)
    r = subprocess.run(["/usr/bin/g++", "-std=c++17", "-Wall", "-O1", "-I" + os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, f"failed checks (bit mask): {r.stdout}"
