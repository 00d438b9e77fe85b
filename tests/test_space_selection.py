"""Host-side pieces of the per-robot force / moment spaces (osc_mft_parametrize_spaces_batched), compiled for the host: the
pure-motion decision that keeps a per-robot task on the MOTION kernels while every robot is free, the reset rule
(parametrize*: Eigen's isApprox of the normalised axes) that the host and the kernels share, the mode word, the validation of
per-robot values, and the new entry points of the library.  No GPU needed."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
CUDA_INC = "/usr/local/cuda/include"
SPS_FORCE_DIM, SPS_MOMENT_DIM, SPS_CL_FORCE, SPS_CL_MOMENT = 1, 2, 4, 8
SPC_BAD_DIM, SPC_BAD_AXIS, SPC_BAD_FLAG, SPC_NONZERO = 1, 2, 4, 8


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    if not os.path.exists(os.path.join(CUDA_INC, "cuda_runtime.h")):
        pytest.skip("CUDA headers not installed")
    out = tmp_path_factory.mktemp("spaces") / "libspace_select_probe.so"
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-fPIC", "-shared", "-I", CUDA_INC, "-o", str(out),
                           os.path.join(HERE, "cpp", "space_select_probe.cpp")])
    lib = C.CDLL(str(out))
    lib.axis_is_approx.argtypes = [C.POINTER(C.c_double)] * 2
    lib.normalize.argtypes = [C.POINTER(C.c_double)] * 2
    lib.normalize.restype = C.c_double
    lib.check_space.argtypes = [C.c_int, C.c_double, C.c_double, C.c_double]
    return lib


def _d3(v):
    return (C.c_double * 3)(*[float(x) for x in v])


@pytest.mark.parametrize("fdim,mdim,clf,clm,full,vel_sat,expected", [
    (0, 0, 0, 0, 1, 0, 1),
    (1, 0, 0, 0, 1, 0, 0),
    (0, 3, 0, 0, 1, 0, 0),
    (0, 0, 1, 0, 1, 0, 0),
    (0, 0, 0, 1, 1, 0, 0),
    (0, 0, 0, 0, 0, 0, 0),    # partial task
    (0, 0, 0, 0, 1, 1, 0),    # velocity saturation
])
def test_pure_motion_without_a_block_reads_the_parameters(probe, fdim, mdim, clf, clm, full, vel_sat, expected):
    assert probe.pure_motion(0, 0, fdim, mdim, clf, clm, full, vel_sat) == expected


@pytest.mark.parametrize("summary,expected", [
    (0, 1),
    (SPS_FORCE_DIM, 0),
    (SPS_MOMENT_DIM, 0),
    (SPS_CL_FORCE, 0),
    (SPS_CL_MOMENT, 0),
    (SPS_FORCE_DIM | SPS_CL_FORCE, 0),
])
def test_pure_motion_with_a_block_reads_the_summary(probe, summary, expected):
    # the broadcast parameters say force control: with a block, only the summary over the robots counts
    assert probe.pure_motion(1, summary, 1, 2, 1, 1, 1, 0) == expected
    assert probe.pure_motion(1, summary, 0, 0, 0, 0, 0, 0) == 0      # partial task
    assert probe.pure_motion(1, summary, 0, 0, 0, 0, 1, 1) == 0      # velocity saturation


def test_reset_rule(probe):
    a = np.array([0.3, -0.2, 0.9])
    u = (C.c_double * 3)()
    assert probe.normalize(_d3(a), u) == pytest.approx(np.linalg.norm(a), rel=1e-15)
    stored = np.array(u[:])
    for axis, same in [(a, True), (2.5 * a, True), (a + 1e-13 * np.array([1, -1, 0.5]), True),
                       (a + 1e-6 * np.array([1, -1, 0.5]), False), (-a, False)]:
        v = (C.c_double * 3)()
        probe.normalize(_d3(axis), v)
        assert probe.axis_is_approx(v, _d3(stored)) == int(same), axis
    probe.normalize(_d3([0, 0, 1]), u)
    assert probe.axis_is_approx(u, _d3([0, 0, 0])) == 0      # a zero stored axis (never parametrised) is never approx
    nan = (C.c_double * 3)(math.nan, 0, 1)
    assert probe.axis_is_approx(nan, _d3([0, 0, 1])) == 0


def test_mode_word(probe):
    for f in range(4):
        for m in range(4):
            for cf in (0, 1):
                for cm in (0, 1):
                    w = probe.mode_word(f, m, cf, cm)
                    assert w & 3 == f and (w >> 2) & 3 == m and bool(w & 16) == bool(cf) and bool(w & 32) == bool(cm)
                    assert (w == 0) == (f == 0 and m == 0 and not cf and not cm)


def test_validation_of_per_robot_values(probe):
    assert probe.check_space(0, math.nan, 0, 0) == 0                 # the axis of dimension 0 / 3 is not read
    assert probe.check_space(3, 0, 0, 0) == SPC_NONZERO
    assert probe.check_space(1, 0, 0, 1) == SPC_NONZERO
    assert probe.check_space(2, 0, 0.02, 0) == SPC_NONZERO
    assert probe.check_space(1, 0, 0.005, 0) == SPC_BAD_AXIS
    assert probe.check_space(2, math.nan, 0, 1) == SPC_BAD_AXIS
    assert probe.check_space(1, math.inf, 0, 1) == SPC_BAD_AXIS
    assert probe.check_space(4, 0, 0, 1) == SPC_BAD_DIM
    assert probe.check_space(-1, 0, 0, 1) == SPC_BAD_DIM
    assert [probe.check_flag(f) for f in (0, 1, 2, -1)] == [0, SPC_NONZERO, SPC_BAD_FLAG, SPC_BAD_FLAG]


def test_entry_points_are_exported_and_the_abi_is_bumped():
    from sai_primitives_b200 import capi
    lib = capi.load_library()
    for name in ("osc_mft_parametrize_spaces_batched", "osc_mft_set_closed_loop_batched", "osc_mft_get_spaces"):
        assert hasattr(lib, name)
    assert lib.osc_abi_version() == 2
