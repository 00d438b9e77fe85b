#!/usr/bin/env python
"""Cost of per-robot force / moment spaces (osc_mft_parametrize_spaces_batched), handles alternating in one process.  Cycles are
enqueued back to back with stepDevice (device-resident q, dq, tau); each window runs for about --seconds and ends in a device
synchronisation, and is repeated --reps times per handle, the order alternating.  Cases:
  free    config 2 (Panda, full six-dof MotionForceTask + JointTask), every robot free: broadcast vs per-robot (same kernel);
  contact config 2, force space dimension 1 along z with closed-loop force control: broadcast with every robot in contact vs
          per-robot with 1 robot and with 50 % of the robots in contact;
  config3 config 3 (partial XYZ task, force dimension 1, closed-loop force, passivity): broadcast vs per-robot identical rows
          vs per-robot random normals.
Prints one JSON line per case and writes them to --out, with the card name and power limit read in the same run.
usage: python tools/bench_per_robot_spaces.py [--n2 65536] [--n3 262144] [--seconds 1.0] [--reps 3] [--out FILE]"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tools.bench_per_robot_gains import card  # noqa: E402

XYZ = [(1, 0, 0), (0, 1, 0), (0, 0, 1)]


def build(sp, q, dq, hier, mode, contact=None):
    """mode: 'broadcast' or 'per_robot'; contact: None (free), a boolean mask of robots in contact, or 'random' normals"""
    from tests.osc_testlib import TASK_POINTS
    N = q.shape[0]
    link, pt = TASK_POINTS["panda"]
    robot = sp.BatchedRobot("panda", N)
    robot.setQ(q); robot.setDq(dq); robot.updateModel()
    dirs = () if hier == 2 else (XYZ, [])
    mft = sp.MotionForceTask(robot, link, (np.eye(3), np.array(pt)), *dirs); jt = sp.JointTask(robot)
    mft.disableInternalOtg(); jt.disableInternalOtg()
    ctrl = sp.RobotController(robot, [mft, jt])
    mft.setGoalPosition(mft.getCurrentPosition() + np.array([0.02, -0.01, 0.01])); jt.setGoalPosition(q + 0.05)
    mft.setGoalForce(np.array([0, 0, -5.0]))
    mft.updateSensedForceAndMoment(np.tile([0, 0, -4.0], (N, 1)), np.zeros((N, 3)))
    if hier == 3:
        mft.enablePassivity()
    z = np.tile([0.0, 0.0, 1.0], (N, 1))
    if mode == "broadcast":
        if contact is not None:
            mft.parametrizeForceMotionSpaces(1, (0, 0, 1)); mft.setClosedLoopForceControl(True)
    elif contact is None:
        mft.parametrizeForceMotionSpaces(np.zeros(N, np.int32), z); mft.setClosedLoopForceControl(np.zeros(N, bool))
    elif isinstance(contact, str):
        rng = np.random.default_rng(5)
        n = rng.normal(size=(N, 3)); n[:, 2] = np.abs(n[:, 2]) + 1.0
        mft.parametrizeForceMotionSpaces(np.ones(N, np.int32), n); mft.setClosedLoopForceControl(np.ones(N, bool))
    else:
        mft.parametrizeForceMotionSpaces(contact.astype(np.int32), z); mft.setClosedLoopForceControl(contact)
    return robot, ctrl


def window(robot, ctrl, d_q, d_dq, d_tau, seconds, per_cycle_ms):
    n = max(50, int(seconds * 1e3 / max(per_cycle_ms, 1e-3)))
    robot.sync()
    t0 = time.perf_counter()
    for _ in range(n):
        ctrl.stepDevice(d_q.data_ptr(), d_dq.data_ptr(), d_tau.data_ptr())
    robot.sync()
    return n, time.perf_counter() - t0


def run_case(name, N, handles, d, seconds, reps, info):
    est = {}
    for m, (robot, ctrl) in handles.items():   # warm-up, then the cycle time that sizes the windows
        est[m] = 1.0
        for _ in range(3):
            n, wall = window(robot, ctrl, *d, 0.3, est[m])
            est[m] = wall / n * 1e3
    names = list(handles)
    rates = {m: [] for m in names}
    for r in range(reps):
        for m in (names if r % 2 == 0 else names[::-1]):
            robot, ctrl = handles[m]
            n, wall = window(robot, ctrl, *d, seconds, est[m])
            rates[m].append(n * N / wall)
    med = {m: float(np.median(v)) for m, v in rates.items()}
    line = {"case": name, "n_robots": N, "robot_cycles_per_s_median": med, "runs": rates,
            "ratio_over_first": {m: med[m] / med[names[0]] for m in names}, "card": info}
    print(json.dumps(line), flush=True)
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n2", type=int, default=65536)
    ap.add_argument("--n3", type=int, default=262144)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import sai_primitives_b200 as sp
    from tests.osc_testlib import sample_states
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs the GPU")
    info = card()
    dev = torch.device("cuda", 0)
    lines = []
    for hier, N in ((2, a.n2), (3, a.n3)):
        base_q, base_dq, _ = sample_states("panda", 1024, min_sigma_ratio=0.1, dirs=None if hier == 2 else np.eye(6)[:, :3])
        pick = np.random.default_rng(11).integers(0, 1024, N)
        q, dq = base_q[pick], base_dq[pick]
        d = (torch.from_numpy(np.ascontiguousarray(q.T)).to(dev), torch.from_numpy(np.ascontiguousarray(dq.T)).to(dev),
             torch.empty((7, N), dtype=torch.float64, device=dev))
        if hier == 2:
            h = {"broadcast": build(sp, q, dq, 2, "broadcast"), "per_robot": build(sp, q, dq, 2, "per_robot")}
            lines.append(run_case("config2_free", N, h, d, a.seconds, a.reps, info)); del h
            one = np.zeros(N, bool); one[N // 3] = True
            half = np.zeros(N, bool); half[::2] = True
            h = {"broadcast_all_contact": build(sp, q, dq, 2, "broadcast", True), "per_robot_1_contact": build(sp, q, dq, 2, "per_robot", one),
                 "per_robot_half_contact": build(sp, q, dq, 2, "per_robot", half)}
            lines.append(run_case("config2_contact", N, h, d, a.seconds, a.reps, info)); del h
        else:
            h = {"broadcast": build(sp, q, dq, 3, "broadcast", True), "per_robot_identical": build(sp, q, dq, 3, "per_robot", np.ones(N, bool)),
                 "per_robot_random_normals": build(sp, q, dq, 3, "per_robot", "random")}
            lines.append(run_case("config3", N, h, d, a.seconds, a.reps, info)); del h
    if a.out:
        with open(a.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
