"""The oracle's restated arithmetic against the REFERENCE'S OWN SOURCE LINES, bit for bit.

oracle/_ref/liboracle_refmath.so holds include/pointcloud.h:126-158 (ComputeCovariance), :194-288 (ComputeEigenvector0/1),
:378-463 (FastEigen3x3_EV) and include/g2o_tools.h:58-69,105-140,149-183 (skew, Sim3Exp<T>, SE3Exp<T>) cut out of
the reference's sources and compiled verbatim against a stand-in for the Eigen types they use (oracle/ref_shim_eigen.hpp).
This pins the restatement (oracle_math.hpp) mechanically: any drift from the reference's text shows up here.

The restatement is compared with the stored results of tests/golden/pin/refmath.npz (made by
tests/golden/pin/make_pin_golden.py, whose seeded inputs the tests rebuild; `backend` names what produced them)
and, where the library is built, with it live."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "pin")
sys.path.insert(0, GOLDEN)
import make_pin_golden as M  # noqa: E402

_dp = C.POINTER(C.c_double)


@pytest.fixture(scope="module")
def stored(oracle_mod):
    g = np.load(os.path.join(GOLDEN, "refmath.npz"))
    inputs = M.refmath_inputs()
    assert oracle_mod.digest(*inputs) == int(g["input_digest"]), "the seeded inputs changed"
    return g, inputs


def _d(a):
    return a.ctypes.data_as(_dp)


def test_covariance_and_smallest_eigenvector_bit_exact(stored, oracle_mod):
    g, (Pall, idxall, off, kinds, _) = stored
    port = oracle_mod.load("port")
    refm = oracle_mod.load_refmath()
    assert (kinds == 0).any() and (kinds == 1).any()   # near a plane (the common case on LiDAR scans), general position
    for trial in range(len(off) - 1):
        P = np.ascontiguousarray(Pall[off[trial]:off[trial + 1]])
        idx = np.ascontiguousarray(idxall[off[trial]:off[trial + 1]])
        m = len(idx)
        cov_port, ev_port = np.zeros(6), np.zeros(3)
        port.orc_covariance(_d(P), idx.ctypes.data_as(C.POINTER(C.c_uint32)), m, _d(cov_port))
        port.orc_smallest_eigvec(_d(cov_port), _d(ev_port))
        assert np.array_equal(cov_port, g["cov"][trial]), trial
        assert np.array_equal(ev_port, g["ev"][trial]), (trial, ev_port, g["ev"][trial])
        if refm is not None:
            cov_ref = np.zeros(9)
            refm.refm_covariance(_d(P), m, idx.ctypes.data_as(C.POINTER(C.c_uint32)), m, _d(cov_ref))
            full = cov_ref.reshape(3, 3)
            assert np.array_equal(full, full.T)
            assert np.array_equal(cov_port, full[np.triu_indices(3)]), trial
            ev_ref, eval_ref = np.zeros(3), np.zeros(3)
            refm.refm_fast_eigen(_d(cov_ref), _d(ev_ref), _d(eval_ref))
            assert np.array_equal(ev_port, ev_ref), (trial, ev_port, ev_ref)


def test_sim3exp_se3exp_bit_exact_including_jets(stored, oracle_mod):
    """Sim3Exp values AND all 7 partials of R, t, s (the dual), and SE3Exp(-x[0:6])."""
    g, (_, _, _, _, xs) = stored
    port = oracle_mod.load("port")
    refm = oracle_mod.load_refmath()
    assert (np.abs(xs[:, :3]).max(axis=1) < 1e-4).any()   # the Taylor branch (theta < 1e-4) is exercised
    for trial, x in enumerate(xs):
        got = M.sim3_se3(port, "orc_", x)
        assert got[2][0] == x[6]
        assert oracle_mod.digest(*got) == int(g["exp"][trial]), trial
        if refm is not None:
            want = M.sim3_se3(refm, "refm_", x)
            assert all(np.array_equal(a, b) for a, b in zip(got, want)), trial
