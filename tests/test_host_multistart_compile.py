"""The multi-start adapter of include/stlcalib_host.hpp (stl::Context::associate_multi / linearize_multi / step_multi,
stl::LMProblemSet) compiles against the C-ABI header (no GPU, no link)."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SRC = r"""
#include "stlcalib_host.hpp"
double use(stl::Context &ctx) {
    stl::LMProblemSet set(ctx);
    const double X0[2][7] = {};
    const uint8_t mask[2] = {1, 0};
    const int32_t prob[3] = {0, 1, 1};
    auto n = set.build(&X0[0][0], 2);
    n = set.build(&X0[0][0], 2, mask);
    const double X[3][7] = {};
    std::vector<stl_lin_sums_t> L = set.evaluate(&X[0][0], 3, prob);
    std::vector<stl_step_sums_t> S = ctx.step_multi(&X0[0][0], 2, mask);
    return L[0].cost + S[1].lin.cost + (double)n[1][0] + set.size();
}
"""


def test_multistart_adapter_compiles(tmp_path):
    src = tmp_path / "multistart.cpp"
    src.write_text(SRC)
    r = subprocess.run(["/usr/bin/g++", "-std=c++17", "-Wall", "-fsyntax-only", "-I" + os.path.join(ROOT, "include"), str(src)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
