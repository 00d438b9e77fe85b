"""Per-robot gains through the C++ host mirror (include/sai_b200/sai_primitives_batched.hpp): build the demo with g++, run it
on the GPU, compare with the oracle, each oracle robot carrying the gains of its GPU robot."""
import os
import subprocess

import numpy as np
import pytest

from tests.osc_testlib import REL_TOL, TASK_POINTS, OracleBatch, rel_err, rng_for, sample_states

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def test_cpp_mirror_per_robot_gains(tmp_path):
    exe = tmp_path / "per_robot_gains_demo"
    libdir = os.path.join(ROOT, "sai_primitives_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "per_robot_gains_demo.cpp"), "-o", str(exe),
                           "-L", libdir, "-lsai_b200_osc", "-Wl,-rpath," + libdir])
    N = 64
    q, dq, _ = sample_states("panda", N, min_sigma_ratio=0.08)
    G = [np.zeros((N, 3)) for _ in range(6)] + [np.zeros((N, 7)) for _ in range(3)]
    lo_hi = [(50, 200), (10, 30), (0.5, 5), (100, 300), (15, 35), (0.5, 5), (20, 100), (5, 20), (0.5, 3)]
    for i in range(N):
        g = rng_for(i, stream=46)
        for a, (lo, hi) in zip(G, lo_hi):
            a[i] = g.uniform(lo, hi, a.shape[1])
    state = tmp_path / "state.bin"
    with open(state, "wb") as f:
        f.write(np.ascontiguousarray(q.T).tobytes()); f.write(np.ascontiguousarray(dq.T).tobytes())
    gains = tmp_path / "gains.bin"
    with open(gains, "wb") as f:
        for a in G:
            f.write(np.ascontiguousarray(a.T).tobytes())
    out = tmp_path / "tau.bin"
    r = subprocess.run([str(exe), str(state), str(gains), str(N), str(out)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)
    assert "0 unhandled" in r.stdout
    tau = np.fromfile(out, dtype=np.float64).reshape(7, N).T
    link, pt = TASK_POINTS["panda"]
    ob = OracleBatch("panda", N); ob.set_state(q, dq)
    omft = ob.add_mft(link, (np.eye(3), np.array(pt))); ojt = ob.add_jt(); ob.finalize()
    for i, (a, b) in enumerate(zip(omft, ojt)):
        a.setPosControlGains(G[0][i], G[1][i], G[2][i]); a.setOriControlGains(G[3][i], G[4][i], G[5][i])
        b.setGains(G[6][i], G[7][i], G[8][i])
        a.setGoalLinearVelocity((0.01, -0.02, 0.03)); b.setGoalVelocity(np.full(7, 0.1))
    for _ in range(3):
        ref = ob.cycle()
    assert rel_err(tau, ref).max() < REL_TOL
