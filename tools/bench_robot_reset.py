#!/usr/bin/env python
"""Cost of per-robot resets (osc_reset_robots) on config 2 (Panda, full six-dof MotionForceTask + JointTask in its null space),
with the internal OTG off and on:
  * the device time of one osc_reset_robots call (device mask) with 0 %, 1 % and 100 % of the robots selected, in both modes,
    from CUDA events around --calls back-to-back calls on the handle's stream;
  * the control rate of a device-resident closed loop (stepDevice + osc_sim_integrate, plus a 1 % construct reset every cycle)
    against the same loop without the reset call, the two alternating, each window about --seconds and ending in a device
    synchronisation.  The state is restored before each window.

Prints one JSON line per (batch size, OTG) with the card name and power limit read in the same run.
usage: python tools/bench_robot_reset.py [--sizes 65536,1048576] [--seconds 1.0] [--reps 3] [--calls 200] [--out FILE]"""
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


def build(sp, q, dq, otg):
    from tests.osc_testlib import TASK_POINTS
    link, pt = TASK_POINTS["panda"]
    robot = sp.BatchedRobot("panda", q.shape[0])
    robot.setQ(q); robot.setDq(dq); robot.updateModel()
    mft = sp.MotionForceTask(robot, link, (np.eye(3), np.array(pt))); jt = sp.JointTask(robot)
    if otg:
        mft.enableInternalOtgAccelerationLimited(0.3, 2.0, np.pi / 3, 2 * np.pi); jt.enableInternalOtgAccelerationLimited(np.pi / 3, 2 * np.pi)
    else:
        mft.disableInternalOtg(); jt.disableInternalOtg()
    ctrl = sp.RobotController(robot, [mft, jt])
    ctrl.enableGravityCompensation(True)
    mft.setPosControlGains(125.0, 20.0, 2.5); mft.setOriControlGains(200.0, 25.0, 2.5); jt.setGains(60.0, 12.0, 1.5)
    mft.setGoalPosition(mft.getCurrentPosition() + np.array([0.02, -0.01, 0.01])); jt.setGoalPosition(q + 0.05)
    return robot, ctrl


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="65536,1048576")
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import sai_primitives_b200 as sp
    from sai_primitives_b200 import capi
    from tests.osc_testlib import sample_states
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs the GPU")
    lib = capi.load_library()
    info = card()
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream()   # the handles run on it (osc_set_stream), so the events below bracket their work
    torch.cuda.set_stream(stream)
    bq, bdq, _ = sample_states("panda", 1024, min_sigma_ratio=0.1)
    lines = []
    for N in [int(s) for s in a.sizes.split(",") if s]:
        pick = np.random.default_rng(11).integers(0, 1024, N)
        q, dq = bq[pick], bdq[pick]
        q0 = torch.from_numpy(np.ascontiguousarray(q.T)).to(dev); dq0 = torch.from_numpy(np.ascontiguousarray(dq.T)).to(dev)
        d_q, d_dq = q0.clone(), dq0.clone()
        d_tau = torch.zeros((7, N), dtype=torch.float64, device=dev)
        rng = np.random.default_rng(5)
        masks = {f: torch.from_numpy((rng.random(N) < f).astype(np.int32) if 0 < f < 1 else np.full(N, int(f), np.int32)).to(dev)
                 for f in (0.0, 0.01, 1.0)}
        for otg in (False, True):
            robot, ctrl = build(sp, q, dq, otg)
            robot.setStream(stream.cuda_stream)
            h = robot.handle
            ctrl.stepDevice(d_q.data_ptr(), d_dq.data_ptr(), d_tau.data_ptr())
            # ---- one reset call
            calls = {}
            for mode, mname in ((capi.OSC_RESET_REINITIALIZE, "reinitialize"), (capi.OSC_RESET_CONSTRUCT, "construct")):
                for f, m in masks.items():
                    ms = []
                    for r in range(a.reps + 1):
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record(stream)
                        for _ in range(a.calls):
                            assert lib.osc_reset_robots(h, -1, m.data_ptr(), capi.OSC_MEM_DEVICE, mode) == 0
                        e1.record(stream)
                        e1.synchronize()
                        if r > 0:   # the first pass warms up
                            ms.append(e0.elapsed_time(e1) / a.calls)
                    calls["%s_%g%%" % (mname, 100 * f)] = {"us_per_call_median": 1e3 * float(np.median(ms)), "us_per_call": [1e3 * x for x in ms]}
            # ---- closed loop with and without a 1 % construct reset every cycle
            m1 = masks[0.01].data_ptr()

            def window(with_reset, n):
                d_q.copy_(q0); d_dq.copy_(dq0)
                robot.setStateDevice(d_q.data_ptr(), d_dq.data_ptr())
                ctrl.reinitializeTasks()
                robot.sync()
                t0 = time.perf_counter()
                for _ in range(n):
                    ctrl.stepDevice(d_q.data_ptr(), d_dq.data_ptr(), d_tau.data_ptr())
                    lib.osc_sim_integrate(h, d_q.data_ptr(), d_dq.data_ptr(), d_tau.data_ptr(), 0.001, 1, capi.OSC_MEM_DEVICE)
                    if with_reset:
                        lib.osc_reset_robots(h, -1, m1, capi.OSC_MEM_DEVICE, capi.OSC_RESET_CONSTRUCT)
                robot.sync()
                return time.perf_counter() - t0

            est = {}
            for v in (False, True):   # warm-up and cycle-time estimate
                window(v, 50)
                est[v] = window(v, 100) / 100
            loop = {False: [], True: []}
            for r in range(a.reps):
                for v in ((False, True) if r % 2 == 0 else (True, False)):
                    n = max(100, int(a.seconds / est[v]))
                    wall = window(v, n)
                    loop[v].append({"cycles": n, "seconds": wall, "robot_cycles_per_s": n * N / wall})
            rate = {v: float(np.median([x["robot_cycles_per_s"] for x in loop[v]])) for v in loop}
            line = {"n_robots": N, "otg": otg, "reset_call": calls,
                    "loop_without_reset": {"robot_cycles_per_s_median": rate[False], "runs": loop[False]},
                    "loop_with_1pct_reset": {"robot_cycles_per_s_median": rate[True], "runs": loop[True]},
                    "ratio_with_over_without": rate[True] / rate[False], "card": info}
            print(json.dumps(line), flush=True)
            lines.append(line)
            robot.close()
    if a.out:
        with open(a.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
