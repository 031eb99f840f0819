"""The keyframe-selection adapter of include/stlcalib_host.hpp (stl::Context::select_keyframes / select_all / eval_frames)
compiles against the C-ABI header (no GPU, no link)."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SRC = r"""
#include "stlcalib_host.hpp"
double use(stl::Context &ctx) {
    ctx.select_keyframes({0, 2, 5});
    const double X[2][7] = {};
    std::vector<double> per_kf = ctx.eval_frames(&X[0][0], 2, 6);
    ctx.select_keyframes({});
    ctx.select_all();
    return per_kf[13 * 6 + 5];
}
"""


def test_select_adapter_compiles(tmp_path):
    src = tmp_path / "select.cpp"
    src.write_text(SRC)
    r = subprocess.run(["/usr/bin/g++", "-std=c++17", "-Wall", "-fsyntax-only", "-I" + os.path.join(ROOT, "include"), str(src)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
