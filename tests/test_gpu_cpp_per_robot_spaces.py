"""Per-robot force spaces and closed-loop flags through the C++ host mirror (include/sai_b200/sai_primitives_batched.hpp): build
the demo with g++, run it on the GPU, compare with the oracle, each oracle robot parametrised like its GPU robot."""
import os
import subprocess

import numpy as np
import pytest

from tests.osc_testlib import REL_TOL, TASK_POINTS, OracleBatch, rel_err, rng_for, sample_states

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def test_cpp_mirror_per_robot_spaces(tmp_path):
    exe = tmp_path / "per_robot_spaces_demo"
    libdir = os.path.join(ROOT, "sai_primitives_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "per_robot_spaces_demo.cpp"), "-o", str(exe),
                           "-L", libdir, "-lsai_b200_osc", "-Wl,-rpath," + libdir])
    N = 64
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.08)
    dims = np.arange(N) % 4
    flags = (np.arange(N) // 4) % 2
    axes = np.array([rng_for(i, stream=47).normal(size=3) for i in range(N)])
    force = np.array([[0, 0, -5.0] + rng_for(i, stream=48).normal(0, 1.0, 3) for i in range(N)])
    state = tmp_path / "state.bin"
    with open(state, "wb") as f:
        f.write(np.ascontiguousarray(q.T).tobytes()); f.write(np.ascontiguousarray(dq.T).tobytes())
    spaces = tmp_path / "spaces.bin"
    with open(spaces, "wb") as f:
        f.write(dims.astype(np.float64).tobytes()); f.write(flags.astype(np.float64).tobytes())
        f.write(np.ascontiguousarray(axes.T).tobytes()); f.write(np.ascontiguousarray(force.T).tobytes())
    out = tmp_path / "tau.bin"
    r = subprocess.run([str(exe), str(state), str(spaces), str(N), str(out)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)
    assert "0 unhandled" in r.stdout
    tau = np.fromfile(out, dtype=np.float64).reshape(7, N).T
    link, pt = TASK_POINTS["panda"]
    ob = OracleBatch("panda", N); ob.set_state(q, dq)
    omft = ob.add_mft(link, (np.eye(3), np.array(pt))); ob.add_jt(); ob.finalize()
    for i, a in enumerate(omft):
        a.setForceControlGains(0.8, 12.0, 1.5); a.setGoalForce((0, 0, -5.0))
        a.parametrizeForceMotionSpaces(int(dims[i]), axes[i]); a.setClosedLoopForceControl(bool(flags[i]))
        a.updateSensedForceAndMoment(force[i], np.zeros(3))
    for _ in range(3):
        ref = ob.cycle()
    assert rel_err(tau, ref).max() < REL_TOL
