"""Host-side decisions of the kernel launcher (csrc/osc_launch.h) about per-robot gains (osc_set_gains), compiled for the host:
a launch reads gain blocks when a leading task has one, and the specialised fused kernel has per-robot instantiations for the
pure-motion full six-dof task and the three-direction task only (every other case takes the non-specialised kernel, which
tests the block pointers at run time).  No GPU needed: the functions only look at the program struct."""
import ctypes as C
import os
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
CUDA_INC = "/usr/local/cuda/include"


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    if not os.path.exists(os.path.join(CUDA_INC, "cuda_runtime.h")):
        pytest.skip("CUDA headers not installed")
    out = tmp_path_factory.mktemp("gains") / "libgain_select_probe.so"
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-fPIC", "-shared", "-I", CUDA_INC, "-o", str(out),
                           os.path.join(HERE, "cpp", "gain_select_probe.cpp")])
    return C.CDLL(str(out))


@pytest.mark.parametrize("blocks,has_jt,jt_first,expected", [
    (0, 1, 0, 0),    # broadcast gains everywhere
    (1, 1, 0, 1),    # motion-force task per robot
    (2, 1, 0, 1),    # joint task per robot
    (3, 1, 0, 1),
    (2, 0, 0, 0),    # a joint-task block does not count when no joint task closes the hierarchy
    (2, 1, 1, 1),    # joint task leading, its block counts
    (1, 0, 1, 0),    # a motion-force task that does not lead the hierarchy is not the specialised kernel's task
])
def test_per_robot_gains_gate(probe, blocks, has_jt, jt_first, expected):
    assert probe.per_robot_case(blocks, has_jt, jt_first) == expected


@pytest.mark.parametrize("R,spec,motion,expected", [
    (6, 1, 1, 1),    # flagship: pure motion control, full six-dof task
    (6, 1, 0, 0),    # force / moment control or velocity saturation: non-specialised kernel
    (6, 0, 0, 0),
    (3, 1, 0, 1),    # three controlled directions, any control law
    (3, 0, 0, 0),
    (5, 1, 0, 0),
    (0, 1, 0, 0),
])
def test_per_robot_specialisations(probe, R, spec, motion, expected):
    assert probe.prg_specialised(R, spec, motion) == expected
