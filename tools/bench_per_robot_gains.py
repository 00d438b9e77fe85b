#!/usr/bin/env python
"""Cost of per-robot PID gains (osc_set_gains) on config 2 (Panda, full six-dof MotionForceTask + JointTask in its null space):
the same handle geometry in broadcast mode and in per-robot mode (every robot with its own position, orientation and joint
gains), alternating in one process.  Cycles are enqueued back to back with stepDevice (device-resident q, dq, tau), each
window runs for about --seconds and ends in a device synchronisation; the window is repeated --reps times per mode.

Prints one JSON line per (batch size, states, mode) and a summary line with the card name and power limit read in the same run.
usage: python tools/bench_per_robot_gains.py [--sizes 65536,1048576] [--unfiltered 131072] [--seconds 1.0] [--reps 3] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split("\n")[0]
        name, plim, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": plim, "max_sm_clock": clk}
    except Exception as e:  # noqa: BLE001  (reported, not hidden)
        return {"error": str(e)}


def build(sp, q, dq, per_robot):
    from tests.osc_testlib import TASK_POINTS
    N = q.shape[0]
    link, pt = TASK_POINTS["panda"]
    robot = sp.BatchedRobot("panda", N)
    robot.setQ(q); robot.setDq(dq); robot.updateModel()
    mft = sp.MotionForceTask(robot, link, (np.eye(3), np.array(pt))); jt = sp.JointTask(robot)
    mft.disableInternalOtg(); jt.disableInternalOtg()
    ctrl = sp.RobotController(robot, [mft, jt])
    rng = np.random.default_rng(3)
    if per_robot:
        mft.setPosControlGains(rng.uniform(50, 200, (N, 3)), rng.uniform(10, 30, (N, 3)), rng.uniform(0.5, 5, (N, 3)))
        mft.setOriControlGains(rng.uniform(100, 300, (N, 3)), rng.uniform(15, 35, (N, 3)), rng.uniform(0.5, 5, (N, 3)))
        jt.setGains(rng.uniform(20, 100, (N, 7)), rng.uniform(5, 20, (N, 7)), rng.uniform(0.5, 3, (N, 7)))
    else:
        mft.setPosControlGains(125.0, 20.0, 2.5); mft.setOriControlGains(200.0, 25.0, 2.5); jt.setGains(60.0, 12.0, 1.5)
    mft.setGoalPosition(mft.getCurrentPosition() + np.array([0.02, -0.01, 0.01])); jt.setGoalPosition(q + 0.05)
    return robot, ctrl


def window(robot, ctrl, d_q, d_dq, d_tau, seconds, per_cycle_ms):
    """enqueue about `seconds` worth of cycles, timed on the host clock up to the device synchronisation; then 200 single
    synchronised cycles for the p50 latency"""
    n = max(50, int(seconds * 1e3 / max(per_cycle_ms, 1e-3)))
    robot.sync()
    t0 = time.perf_counter()
    for _ in range(n):
        ctrl.stepDevice(d_q.data_ptr(), d_dq.data_ptr(), d_tau.data_ptr())
    robot.sync()
    wall = time.perf_counter() - t0
    lat = []
    for _ in range(200):
        t = time.perf_counter()
        ctrl.stepDevice(d_q.data_ptr(), d_dq.data_ptr(), d_tau.data_ptr())
        robot.sync()
        lat.append(time.perf_counter() - t)
    return n, wall, float(np.median(lat))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="65536,1048576")
    ap.add_argument("--unfiltered", type=int, default=131072)
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
    cases = [(int(s), True) for s in a.sizes.split(",") if s] + ([(a.unfiltered, False)] if a.unfiltered else [])
    lines = []
    base = {True: sample_states("panda", 1024, min_sigma_ratio=0.1), False: sample_states("panda", 1024)}
    for N, filtered in cases:
        bq, bdq, _ = base[filtered]
        pick = np.random.default_rng(11).integers(0, 1024, N)
        q, dq = bq[pick], bdq[pick]
        d_q = torch.from_numpy(np.ascontiguousarray(q.T)).to(dev); d_dq = torch.from_numpy(np.ascontiguousarray(dq.T)).to(dev)
        d_tau = torch.empty((7, N), dtype=torch.float64, device=dev)
        handles = {m: build(sp, q, dq, m == "per_robot") for m in ("broadcast", "per_robot")}
        est = {}
        for m, (robot, ctrl) in handles.items():   # warm-up: module load, split-path allocation, steady state; then the cycle time
            est[m] = 1.0
            for _ in range(3):
                n, wall, _ = window(robot, ctrl, d_q, d_dq, d_tau, 0.3, est[m])
                est[m] = wall / n * 1e3
        res = {m: [] for m in handles}
        for r in range(a.reps):
            for m in (("broadcast", "per_robot") if r % 2 == 0 else ("per_robot", "broadcast")):
                robot, ctrl = handles[m]
                n, wall, p50 = window(robot, ctrl, d_q, d_dq, d_tau, a.seconds, est[m])
                res[m].append({"cycles": n, "seconds": wall, "robot_cycles_per_s": n * N / wall, "p50_latency_ms": p50 * 1e3})
        summ = {}
        for m, rs in res.items():
            rates = [x["robot_cycles_per_s"] for x in rs]
            summ[m] = {"robot_cycles_per_s_median": float(np.median(rates)), "min": min(rates), "max": max(rates),
                       "p50_latency_ms_median": float(np.median([x["p50_latency_ms"] for x in rs])), "runs": rs}
        line = {"n_robots": N, "states": "filtered" if filtered else "unfiltered", "broadcast": summ["broadcast"], "per_robot": summ["per_robot"],
                "ratio_per_robot_over_broadcast": summ["per_robot"]["robot_cycles_per_s_median"] / summ["broadcast"]["robot_cycles_per_s_median"],
                "card": info}
        print(json.dumps(line), flush=True)
        lines.append(line)
        del handles
    if a.out:
        with open(a.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
