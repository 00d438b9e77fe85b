#!/usr/bin/env python
"""Benchmark of the batched operational-space controller (BASELINE.json metric:
robot control cycles/sec, batched OSC torques; p99 cycle latency).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--robots R] [--impl reference] [--dump-outputs DIR]

A step = one control cycle (kinematics/dynamics -> task models -> torques) for one batch of
R robots per GPU.  Workload (config.workload): BASELINE config 2 -- Panda, MotionForceTask 6-DoF at the
end-effector + JointTask in its null space through RobotController, 65,536 robots per GPU (weak scaling:
robots are sharded by batch index, one process per GPU, no collective on the control path).

  value  whole-job cycles/s with q, dq, goals resident in HBM (device pointers through the C ABI);
  e2e    the same metric through the C ABI with pinned HOST buffers: H2D of q, dq and D2H of tau inside
         the timed region;
  roofline  the fused kernel against the FP64 roofline (SURVEY.md 8d: 9.5 kFLOP per robot-cycle);
  cpu_baseline  the reference's own control law (oracle/_ref/libsai_ref.so: /root/reference/src compiled in place against
         stand-ins for Eigen and sai-model, kind "reference") looped over a bounded sample on the host cores; the plain C++
         port (oracle/cpp) is timed beside it (`port`), and takes over (kind "port") where the library was not built.
--impl reference runs only that CPU arm, on the same 65,536 states as the GPU arm, all host threads.

Timing: after SETUP_ROUNDS set-up cycles of every controller instance (`timing.setup_cycles`) and `--warmup W` cycles,
exactly `--steps K` back-to-back cycles are timed between two CUDA events (barrier + synchronize on both sides);
`ms_per_step` = that time / K.  A 20-step region lasts about 0.7 ms, so small K is noisy.

--dump-outputs DIR writes the torques of the last timed cycle (rank 0's batch) to DIR/tau.npy, float64, in the [dof, robots]
layout osc_step returns; above DUMP_BYTES_MAX a fixed sample of robots is written, with their indices (stored as float64)
in DIR/robot_index.npy.  The inputs depend only on the arguments (seeded), so two builds can be compared output for output.
The benchmark writes nothing into the source tree.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True    # the source tree may be read-only: no __pycache__ for the modules imported below
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "robot_control_cycles_per_sec"
UNIT = "cycles/s"
FLOP_PER_CYCLE = 9.5e3        # SURVEY.md section 8(d), config 2
FP64_PEAK_TFLOPS = 37.2       # 148 SM x 64 FMA/clk x 2 x 1.965 GHz (no FP64 entry in MEASURED_PEAKS.json)
FP32_PEAK_TFLOPS = 74.4       # 148 SM x 128 FMA/clk x 2 x 1.965 GHz (optional FP32 mode, reported separately)
WORKLOAD = "config2: Panda MotionForceTask 6-DoF + JointTask null space via RobotController, OTG off, BIE decoupling (reference defaults)"
ROBOT = "panda"
LINK, POINT = "end-effector", (0.0, 0.0, 0.07)
SEED = 1234
DUMP_BYTES_MAX = 64_000_000   # --dump-outputs: larger outputs are written as a fixed sample of robots
SETUP_ROUNDS = 6              # set-up cycles per controller instance before the warm-up (see gpu_arm)
LATENCY_SAMPLES = 1000        # SURVEY.md 8d: >= 1000 single-cycle brackets for the percentiles


def workload_config(args, world):
    """`config` of the JSON line: the definition of the workload, identical for both arms (measured properties of the
    sampled inputs go under `inputs`)"""
    R = args.robots
    return {"workload": WORKLOAD, "robots_per_gpu": R, "robots_total": R * world,
            "state_filter": "uniform joint states, rejected while s_min/s_max < %.3g (SURVEY.md 8d)" % args.min_ratio,
            "l2": "inputs larger than L2: %d controller instances (%.0f MB of state) used round-robin" % (args.sets, args.sets * R * 8 * 250 / 1e6),
            "parallelism": "robots sharded by batch index, one process per GPU, no collective"}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def dump_outputs(out_dir, tau_of_last_step):
    """--dump-outputs: tau [dof, robots] as DIR/tau.npy; beyond DUMP_BYTES_MAX, a fixed sample of robots (same indices on
    every run with the same arguments) plus DIR/robot_index.npy, the sampled robots' indices in ascending order, stored as
    float64 (exact below 2**53) so that every file of the dump has the same dtype"""
    os.makedirs(out_dir, exist_ok=True)
    tau = np.ascontiguousarray(tau_of_last_step, dtype=np.float64)
    n, R = tau.shape
    if R * n * 8 > DUMP_BYTES_MAX:
        keep = ((DUMP_BYTES_MAX - 4096) // 8) // (n + 1)     # a sampled robot costs n torques + its index; 4 KB for headers
        idx = np.sort(np.random.default_rng(0).choice(R, size=keep, replace=False))
        np.save(os.path.join(out_dir, "robot_index.npy"), idx.astype(np.float64))
        tau = np.ascontiguousarray(tau[:, idx])
    np.save(os.path.join(out_dir, "tau.npy"), tau)
    log("[dump] tau of the last timed cycle, %d x %d float64 -> %s" % (tau.shape[0], tau.shape[1], out_dir))


# ------------------------------------------------------------------ synthetic inputs (SURVEY.md 8d)
def sample_batch(sp, n_robots, device, min_ratio=0.1, shard=0):
    """q ~ U(lo+0.1 range, hi-0.1 range), dq ~ U(-1,1); states whose task Jacobian has
    s_min/s_max < min_ratio are rejected before timing so the timed path is the non-singular one.
    The Jacobians of the candidates come from the library's own kinematics stage (input generation only)."""
    desc = sp.capi.ModelDesc()
    sp.capi.load_library().osc_builtin_model(ROBOT.encode(), C.byref(desc))
    n = desc.n
    lo = np.array(desc.q_lower[:n]); hi = np.array(desc.q_upper[:n])
    rng = np.random.Generator(np.random.Philox(key=SEED + shard))   # counter-based: every shard regenerates its own slice
    q_ok = np.zeros((0, n)); dq_ok = np.zeros((0, n))
    tried = 0
    accepted = 0
    chunk = 131072
    probe = sp.BatchedRobot(ROBOT, chunk, device=device)
    while q_ok.shape[0] < n_robots:
        q = lo + (0.1 + 0.8 * rng.random((chunk, n))) * (hi - lo)
        dq = rng.uniform(-1.0, 1.0, (chunk, n))
        probe.setQ(q); probe.setDq(dq); probe.updateModel()
        J = probe.evalModel(LINK, POINT)["J"]
        w = np.linalg.eigvalsh(J @ J.transpose(0, 2, 1))
        keep = np.sqrt(np.maximum(w[:, 0], 0) / w[:, -1]) >= min_ratio
        q_ok = np.concatenate([q_ok, q[keep]]); dq_ok = np.concatenate([dq_ok, dq[keep]])
        tried += chunk
        accepted += int(keep.sum())
    probe.close()
    q_ok, dq_ok = q_ok[:n_robots], dq_ok[:n_robots]
    return q_ok, dq_ok, 1.0 - accepted / max(tried, 1), rng


def make_goals(rng, x, R, q):
    N, n = q.shape
    def expm(w):
        th = np.linalg.norm(w, axis=1, keepdims=True)
        k = w / np.maximum(th, 1e-12)
        K = np.zeros((N, 3, 3))
        K[:, 0, 1], K[:, 0, 2], K[:, 1, 0], K[:, 1, 2], K[:, 2, 0], K[:, 2, 1] = -k[:, 2], k[:, 1], k[:, 2], -k[:, 0], -k[:, 1], k[:, 0]
        s, c = np.sin(th)[:, :, None], np.cos(th)[:, :, None]
        return np.eye(3)[None] + s * K + (1 - c) * (K @ K)
    return dict(
        xd=x + rng.uniform(-0.05, 0.05, (N, 3)), Rd=R @ expm(rng.uniform(-0.2, 0.2, (N, 3))),
        vd=rng.uniform(-0.1, 0.1, (N, 3)), wd=rng.uniform(-0.1, 0.1, (N, 3)),
        ad=rng.uniform(-0.5, 0.5, (N, 3)), ald=rng.uniform(-0.5, 0.5, (N, 3)),
        qd=q + rng.uniform(-0.2, 0.2, (N, n)))


# ------------------------------------------------------------------ clocks
class ClockSampler:
    QUERY = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "nvidia-smi unavailable"}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [l for (t, l) in self.samples if t0 - 0.05 <= t <= t1 + 0.15] or [l for (_, l) in self.samples]
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in rows:
            f = [x.strip() for x in l.split(",")]
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except Exception:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------ CPU arm
CPU_CHUNK = 8192      # robots per controller batch on the host (70 KB per reference controller instance)


class CpuControllers:
    """A chunk of CPU controllers for config 2, all host threads: the reference's own compiled control law
    (oracle/_ref/libsai_ref.so, kind "reference") when the library exists, else the C++ port (kind "port").
    run(q, dq, goals) pushes any number of robots through it chunk by chunk: per robot and cycle setQ / setDq / updateModel,
    goal setters, updateControllerTaskModels, computeControlTorques -- the reference's user loop."""

    def __init__(self, kind, n_chunk):
        self.kind, self.n_chunk = kind, n_chunk
        comp = (np.eye(3), np.array(POINT))
        if kind == "reference":
            from oracle.sai_ref import RefBatch
            self.b = RefBatch(ROBOT, n_chunk, oriented=False)
            self.b.add_mft(LINK, comp); self.b.add_jt(); self.b.finalize()
            self.tm, self.tj = 0, 1
        else:
            from oracle.cpp_ref import CppOracleBatch
            self.b = CppOracleBatch(ROBOT, n_chunk)
            self.tm = self.b.add_mft(LINK, comp); self.tj = self.b.add_jt()
        self.threads = self.b.hardware_threads()

    def run(self, q, dq, goals):
        N = q.shape[0]
        tau = np.zeros_like(q)
        for lo in range(0, N, self.n_chunk):
            hi = min(N, lo + self.n_chunk)
            idx = np.arange(lo, lo + self.n_chunk) % N if hi - lo < self.n_chunk else slice(lo, hi)   # last chunk padded by wrapping
            g = {k: v[idx] for k, v in goals.items()}
            if self.kind == "reference":
                self.b.mft_set_goals(self.tm, g["xd"], g["Rd"], g["vd"], g["wd"], g["ad"], g["ald"]); self.b.jt_set_goal_positions(self.tj, g["qd"])
            else:
                self.b.mft_set_goals(self.tm, g["xd"], g["Rd"], g["vd"], g["wd"], g["ad"], g["ald"]); self.b.jt_set_goals(self.tj, g["qd"])
            t = self.b.step(q[idx], dq[idx], n_threads=self.threads)
            tau[lo:hi] = t[:hi - lo]
        return tau

    def close(self):
        self.b.close()


def cpu_kind():
    from oracle import sai_ref
    return "reference" if sai_ref.available(oriented=False) else "port"


KIND_TEXT = {"reference": "reference's own RobotController/MotionForceTask/JointTask sources compiled in place (oracle/_ref/libsai_ref.so; "
                          "stand-ins for Eigen and sai-model), -O2",
             "port": "C++ restatement of the reference path (oracle/cpp), -O2"}


def run_cpu_baseline(n_sample, target_seconds, q, dq, goals):
    """bounded sample of the GPU arm's own batch on the host cores; returns {kind: (cycles/s, seconds per run, runs, threads)}"""
    out = {}
    kinds = ["reference", "port"] if cpu_kind() == "reference" else ["port"]
    g = {k: v[:n_sample] for k, v in goals.items()}
    for kind in kinds:
        cc = CpuControllers(kind, min(n_sample, CPU_CHUNK))
        cc.run(q[:n_sample], dq[:n_sample], g)   # warm-up
        times = []
        t_start = time.time()
        while True:
            t0 = time.perf_counter()
            cc.run(q[:n_sample], dq[:n_sample], g)
            times.append(time.perf_counter() - t0)
            if time.time() - t_start > target_seconds / len(kinds) and len(times) >= 3:
                break
        med = float(np.median(times))
        out[kind] = (n_sample / med, med, len(times), cc.threads)
        cc.close()
    return out


def sample_batch_cpu(n_robots, min_ratio, rng):
    """the GPU arm's state distribution without a GPU: vectorised forward kinematics of the Panda in numpy for the
    rejection test (input generation only)"""
    from oracle.robots import make_chain
    ch = make_chain(ROBOT)
    b, R_lb, t_lb = ch.link_frames[LINK]
    p_local = t_lb + R_lb @ np.array(POINT)
    q_ok = np.zeros((0, ch.n)); dq_ok = np.zeros((0, ch.n))
    tried = 0
    while q_ok.shape[0] < n_robots:
        M = 65536
        q = ch.q_lower + (0.1 + 0.8 * rng.random((M, ch.n))) * (ch.q_upper - ch.q_lower)
        dq = rng.uniform(-1.0, 1.0, (M, ch.n))
        R = np.tile(np.eye(3), (M, 1, 1)); p = np.zeros((M, 3))
        axes, origins = [], []
        for i in range(ch.n):
            p = p + R @ ch.t_fix[i]
            R = R @ ch.R_fix[i]
            c, s_ = np.cos(q[:, i]), np.sin(q[:, i])
            Rz = np.zeros((M, 3, 3)); Rz[:, 0, 0] = c; Rz[:, 0, 1] = -s_; Rz[:, 1, 0] = s_; Rz[:, 1, 1] = c; Rz[:, 2, 2] = 1
            R = R @ Rz                    # every Panda joint is revolute about its local z axis
            axes.append(R[:, :, 2].copy()); origins.append(p.copy())
        x = p + R @ p_local
        J = np.zeros((M, 6, ch.n))
        for i in range(ch.n):
            J[:, :3, i] = np.cross(axes[i], x - origins[i]); J[:, 3:, i] = axes[i]
        w = np.linalg.eigvalsh(J @ J.transpose(0, 2, 1))
        keep = np.sqrt(np.maximum(w[:, 0], 0) / w[:, -1]) >= min_ratio
        q_ok = np.concatenate([q_ok, q[keep]]); dq_ok = np.concatenate([dq_ok, dq[keep]])
        tried += M
    return q_ok[:n_robots], dq_ok[:n_robots], 1.0 - q_ok.shape[0] / tried


def reference_arm(args):
    """bench.py --impl reference: the reference's own CPU path on the same workload as the GPU arm (config 2, args.robots
    robots per step, same state filter), all host threads.  No GPU, no product code."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    rng = np.random.Generator(np.random.Philox(key=SEED))
    q, dq, rejected = sample_batch_cpu(args.robots, args.min_ratio, rng)
    goals = goals_from_poses(q, rng)
    kind = cpu_kind()
    cc = CpuControllers(kind, min(args.robots, CPU_CHUNK))
    for _ in range(max(1, min(args.warmup, 2))):
        cc.run(q, dq, goals)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        tau = cc.run(q, dq, goals)
    dt = time.perf_counter() - t0
    if not np.isfinite(tau).all():
        raise SystemExit("bench --impl reference: non-finite torques")
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, tau_of_last_step=tau.T)
    value = args.robots * args.steps / dt
    sample = "%d robots x %d cycles (the GPU arm's config: same robot count per step, same state filter s_min/s_max >= %.3g), %s, %d host threads" \
             % (args.robots, args.steps, args.min_ratio, KIND_TEXT[kind], cc.threads)
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, max(1, args.gpus)),
        "inputs": {"rejected_fraction": rejected, "what": "one rank's shard (%d robots per step) on the host cores" % args.robots},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cc.threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out), flush=True)


def goals_from_poses(q, rng):
    """current pose of every robot by vectorised forward kinematics (same arithmetic as sample_batch_cpu), then the
    SURVEY 8d goal perturbation"""
    from oracle.robots import make_chain
    ch = make_chain(ROBOT)
    b, R_lb, t_lb = ch.link_frames[LINK]
    p_local = t_lb + R_lb @ np.array(POINT)
    N = q.shape[0]
    Rr = np.tile(np.eye(3), (N, 1, 1)); p = np.zeros((N, 3))
    for i in range(ch.n):
        p = p + Rr @ ch.t_fix[i]
        Rr = Rr @ ch.R_fix[i]
        c, s_ = np.cos(q[:, i]), np.sin(q[:, i])
        Rz = np.zeros((N, 3, 3)); Rz[:, 0, 0] = c; Rz[:, 0, 1] = -s_; Rz[:, 1, 0] = s_; Rz[:, 1, 1] = c; Rz[:, 2, 2] = 1
        Rr = Rr @ Rz
    return make_goals(rng, p + Rr @ p_local, Rr @ R_lb, q)


# ------------------------------------------------------------------ host memory placement
def place_host_memory_near_gpu(local_rank):
    """Best effort, before any pinned allocation: prefer host memory (and CPUs) of the NUMA node the GPU hangs off, so that the
    ranks of one box do not all stage their host buffers through one socket.  Returns what was found and done (reported under
    e2e.host_placement); does nothing when the platform hides the topology (numa_node = -1, single node, restricted cpuset)."""
    info = {"gpu_numa_node": None, "nodes_online": None, "mempolicy": "unchanged", "cpus": "unchanged"}
    try:
        bus = subprocess.check_output(["nvidia-smi", "-i", str(local_rank), "--query-gpu=pci.bus_id", "--format=csv,noheader"], text=True).strip().lower()
        if bus.count(":") == 2 and len(bus.split(":")[0]) == 8:
            bus = bus[4:]                                   # sysfs uses a 4-digit domain
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read().strip())
        info["gpu_numa_node"] = node
        info["nodes_online"] = open("/sys/devices/system/node/online").read().strip()
        if node < 0 or info["nodes_online"] in ("0", ""):
            return info
        libc = C.CDLL(None, use_errno=True)
        mask = C.c_ulong(1 << node)
        if libc.syscall(238, 1, C.byref(mask), 64) == 0:    # set_mempolicy(MPOL_PREFERRED, {node})
            info["mempolicy"] = "MPOL_PREFERRED node %d" % node
        else:
            info["mempolicy"] = "set_mempolicy failed (errno %d)" % C.get_errno()
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
            info["cpus"] = "%d cpus of node %d" % (len(allowed), node)
    except Exception as e:
        info["error"] = str(e)[:120]
    return info


# ------------------------------------------------------------------ GPU arm
def gpu_arm(args):
    import torch
    import torch.distributed as dist

    import sai_primitives_b200 as sp
    from sai_primitives_b200 import capi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path (use --impl reference for the CPU arm)")
    placement = place_host_memory_near_gpu(local_rank)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = capi.load_library()
    R = args.robots
    n = 7
    n_sets = args.sets

    # ---- inputs: one accepted batch per rank (different Philox stream per rank), copied into n_sets controller
    # instances so that consecutive steps touch different HBM (total working set > L2)
    global SEED
    SEED = 1234 + rank
    t_gen = time.time()
    q, dq, rejected, rng = sample_batch(sp, R, local_rank, min_ratio=args.min_ratio, shard=rank)
    log("[rank %d] sampled %d non-singular states (rejected fraction %.3f) in %.1fs" % (rank, R, rejected, time.time() - t_gen))

    # a dedicated (non-default) stream shared by torch and the library, so that torch.cuda.Event timing sees the kernels
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    sets = []
    goals = None
    for s in range(n_sets):
        robot = sp.BatchedRobot(ROBOT, R, device=local_rank)
        robot.setStream(stream.cuda_stream)
        robot.setQ(q); robot.setDq(dq); robot.updateModel()
        mft = sp.MotionForceTask(robot, LINK, (np.eye(3), np.array(POINT)))
        jt = sp.JointTask(robot)
        mft.disableInternalOtg(); jt.disableInternalOtg()       # BASELINE config 2: internal OTG off (examples/01-...cpp:136)
        ctrl = sp.RobotController(robot, [mft, jt])
        if goals is None:
            goals = make_goals(rng, mft.getCurrentPosition(), mft.getCurrentOrientation(), q)
        mft.setGoalPosition(goals["xd"]); mft.setGoalOrientation(goals["Rd"]); mft.setGoalLinearVelocity(goals["vd"])
        mft.setGoalAngularVelocity(goals["wd"]); mft.setGoalLinearAcceleration(goals["ad"]); mft.setGoalAngularAcceleration(goals["ald"])
        jt.setGoalPosition(goals["qd"])
        d_q = torch.from_numpy(np.ascontiguousarray(q.T)).to(dev)      # SoA [n, R]
        d_dq = torch.from_numpy(np.ascontiguousarray(dq.T)).to(dev)
        d_tau = torch.zeros((n, R), dtype=torch.float64, device=dev)
        sets.append(dict(robot=robot, ctrl=ctrl, q=d_q, dq=d_dq, tau=d_tau))
    torch.cuda.synchronize()

    def step_device(s):
        rc = lib.osc_step(s["robot"].handle, C.c_void_p(s["q"].data_ptr()), C.c_void_p(s["dq"].data_ptr()),
                          C.c_void_p(s["tau"].data_ptr()), capi.OSC_MEM_DEVICE)
        if rc != 0:
            raise RuntimeError(lib.osc_last_error(s["robot"].handle))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing.  The clock sampler starts first so that the set-up and warm-up cycles, not an idle
    # pause, come right before the timed region.
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
        time.sleep(0.25)
    # set-up: a handle picks its general-path grid from the hand-over counts of completed cycles and needs a few cycles
    # to settle on the small one (osc_capi.cu run_cycle), so every instance runs them here: rounds of one cycle per
    # instance, back to back like the timed region, each round completed before the next
    for _ in range(SETUP_ROUNDS):
        for s_ in sets:
            step_device(s_)
        torch.cuda.synchronize()
    for w in range(args.warmup):
        step_device(sets[w % n_sets])
    barrier()
    t_wall0 = time.time()
    # the timed region: exactly args.steps back-to-back cycles between two CUDA events, nothing else in the stream
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = sum(s["robot"].launchCount() for s in sets)
    barrier()
    e0.record()
    for k in range(args.steps):
        step_device(sets[k % n_sets])
    e1.record()
    barrier()
    total_ms = e0.elapsed_time(e1)
    launches = sum(s["robot"].launchCount() for s in sets) - l0
    t_wall1 = time.time()
    if world > 1:          # the slowest rank
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    if args.dump_outputs and rank == 0:
        # later sections reuse the controller instances: keep what the last timed cycle returned now
        dump_outputs(args.dump_outputs, tau_of_last_step=sets[(args.steps - 1) % n_sets]["tau"].cpu().numpy())
    # latency of a single batched cycle, measured in a second pass: an event between two cycles keeps the next fast
    # kernel from being scheduled behind the general-path kernel (programmatic dependent launch), so the per-cycle
    # brackets are not part of the throughput measurement
    lat_n = max(args.steps, LATENCY_SAMPLES)      # SURVEY.md 8d: >= 1000 timed cycles for the percentiles
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(lat_n)]
    for k in range(lat_n):
        ev[k][0].record()
        step_device(sets[k % n_sets])
        ev[k][1].record()
    barrier()
    per_step_ms = np.array([a.elapsed_time(b) for a, b in ev])
    clk = clocks.stop(t_wall0, t_wall1) if rank == 0 else None

    # parity guard on the timed data: every robot stayed on the fast path and the torques are finite
    st = sets[0]["robot"].status()
    tau_host = sets[0]["tau"].cpu().numpy()
    singular_fraction = float(((st & capi.STATUS_SINGULAR_PATH) != 0).mean())
    if (st & capi.STATUS_UNHANDLED).any() or not np.isfinite(tau_host).all():
        raise SystemExit("bench: robots left the CUDA fast path (%d unhandled)" % int(((st & capi.STATUS_UNHANDLED) != 0).sum()))

    # ---- same device-resident cycles with every controller instance on its own stream: independent batches overlap on
    # the GPU, which fills the SMs the last wave of a 65,536-robot launch leaves idle (reported as an extra, not as value)
    for s_ in sets:
        s_["robot"].setStream(0)          # back to the handle's own non-blocking stream
    def step_own_stream(s_):
        rc = lib.osc_step_async(s_["robot"].handle, C.c_void_p(s_["q"].data_ptr()), C.c_void_p(s_["dq"].data_ptr()),
                                C.c_void_p(s_["tau"].data_ptr()), capi.OSC_MEM_DEVICE)
        if rc != 0:
            raise RuntimeError(lib.osc_last_error(s_["robot"].handle))
    for w in range(n_sets):
        step_own_stream(sets[w])
    for s_ in sets:
        s_["robot"].sync()
    barrier()
    multi_steps = max(args.steps, 400)
    t0 = time.perf_counter()
    for k in range(multi_steps):
        step_own_stream(sets[k % n_sets])
    for s_ in sets:
        s_["robot"].sync()
    multi_ms = 1e3 * (time.perf_counter() - t0)
    barrier()

    # ---- the same hierarchy on UNFILTERED states (about half of the uniformly sampled Panda states sit inside the reference's
    # singularity blending band and leave the fused kernel for the general path): reported as an extra so that the cost of
    # that path is timed by the same run, not part of `value`
    def unfiltered_run(Ru, cycles, shard):
        uq, udq, _, _ = sample_batch(sp, Ru, local_rank, min_ratio=0.0, shard=shard)
        urobot = sp.BatchedRobot(ROBOT, Ru, device=local_rank)
        urobot.setStream(stream.cuda_stream)
        urobot.setQ(uq); urobot.setDq(udq); urobot.updateModel()
        umft = sp.MotionForceTask(urobot, LINK, (np.eye(3), np.array(POINT))); ujt = sp.JointTask(urobot)
        umft.disableInternalOtg(); ujt.disableInternalOtg()
        uctrl = sp.RobotController(urobot, [umft, ujt])
        ug = make_goals(rng, umft.getCurrentPosition(), umft.getCurrentOrientation(), uq)
        umft.setGoalPosition(ug["xd"]); umft.setGoalOrientation(ug["Rd"]); umft.setGoalLinearVelocity(ug["vd"]); umft.setGoalAngularVelocity(ug["wd"])
        ujt.setGoalPosition(ug["qd"])
        ud = dict(robot=urobot, q=torch.from_numpy(np.ascontiguousarray(uq.T)).to(dev), dq=torch.from_numpy(np.ascontiguousarray(udq.T)).to(dev),
                  tau=torch.zeros((n, Ru), dtype=torch.float64, device=dev))
        torch.cuda.set_stream(stream)
        for _ in range(3):
            step_device(ud)
            urobot.sync()     # the host reads the hand-over count of completed cycles: let it settle on the path it will use
        barrier()
        ue0, ue1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ue0.record()
        for _ in range(cycles):
            step_device(ud)
        ue1.record()
        barrier()
        ms = ue0.elapsed_time(ue1) / cycles
        ust = urobot.status()
        share = float(((ust & capi.STATUS_SINGULAR_PATH) != 0).mean())
        if (ust & capi.STATUS_UNHANDLED).any():
            raise SystemExit("bench: unfiltered batch left the CUDA path")
        del uctrl
        urobot.close()
        return ms, share

    unfiltered_ms, unfiltered_singular = unfiltered_run(R, 30, rank + 1000)
    # and at a batch size where the hand-over list is many waves long (the split blending path, DESIGN.md section 6 item 9)
    R_LARGE = 1048576
    unfiltered_large_ms, unfiltered_large_singular = (unfiltered_run(R_LARGE, 10, rank + 2000) if R < R_LARGE else (float("nan"), float("nan")))

    # ---- end to end through the C ABI with pinned HOST buffers: every step copies q, dq host->device and tau
    # device->host inside the timed region.  The n_sets controller instances run on their own streams
    # (osc_step_async), so the copies of one instance overlap the kernels of the others; the region is closed by
    # osc_sync on every instance and timed on the host clock (several streams: no single CUDA-event bracket exists).
    for s_ in sets:
        # q and dq adjacent in one pinned buffer: the library then moves the state in a single host->device copy
        s_["hstate"] = torch.empty((2 * n, R), dtype=torch.float64).pin_memory()
        s_["hq"] = s_["hstate"][:n]; s_["hdq"] = s_["hstate"][n:]
        s_["hq"].copy_(torch.from_numpy(np.ascontiguousarray(q.T))); s_["hdq"].copy_(torch.from_numpy(np.ascontiguousarray(dq.T)))
        s_["htau"] = torch.zeros((n, R), dtype=torch.float64).pin_memory()

    def step_host(s_):
        rc = lib.osc_step_async(s_["robot"].handle, C.c_void_p(s_["hq"].data_ptr()), C.c_void_p(s_["hdq"].data_ptr()),
                                C.c_void_p(s_["htau"].data_ptr()), capi.OSC_MEM_HOST)
        if rc != 0:
            raise RuntimeError(lib.osc_last_error(s_["robot"].handle))

    def sync_all():
        for s_ in sets:
            s_["robot"].sync()

    e2e_steps = 200
    for w in range(max(3, n_sets)):
        step_host(sets[w % n_sets])
    sync_all()
    e2e_runs = []
    for rep in range(3):            # median of three passes of e2e_steps cycles each (PCIe throughput varies between passes)
        barrier()
        t0 = time.perf_counter()
        for k in range(e2e_steps):
            step_host(sets[k % n_sets])
        sync_all()
        e2e_runs.append(1e3 * (time.perf_counter() - t0))
    e2e_ms = float(np.median(e2e_runs))
    barrier()
    checksum = float(sum(float(s_["htau"].sum()) for s_ in sets))
    ref_tau = sets[0]["tau"].cpu()
    if not torch.equal(sets[0]["htau"], ref_tau):
        raise SystemExit("bench: end-to-end torques differ from the device-resident run")

    # ---- what the host link gives: the same bytes per step (q, dq in, tau out) as plain pinned cudaMemcpyAsync copies with
    # no kernel at all, host->device and device->host on two streams at once; the end-to-end number is bounded by it
    s1, s2 = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    d_in = torch.empty((2 * n, R), dtype=torch.float64, device=dev); d_out = torch.zeros((n, R), dtype=torch.float64, device=dev)
    def copies(count):
        for _ in range(count):
            with torch.cuda.stream(s1):
                d_in.copy_(sets[0]["hstate"], non_blocking=True)
            with torch.cuda.stream(s2):
                sets[0]["htau"].copy_(d_out, non_blocking=True)
        s1.synchronize(); s2.synchronize()
    copies(10)
    barrier()
    t0 = time.perf_counter()
    copies(100)
    link_ms = 1e3 * (time.perf_counter() - t0) / 100
    barrier()
    sets[0]["htau"].copy_(ref_tau)

    # ---- measured FP64 FMA rate of this GPU (rank 0): the datasheet-derived 37.2 TFLOP/s stays the roofline denominator,
    # the measured figure is reported next to it
    fp64_measured = None
    if rank == 0:
        t_ = C.c_double(0.0)
        if lib.osc_measure_fp64_peak(sets[0]["robot"].handle, C.c_double(0.4), C.byref(t_)) == 0:
            fp64_measured = float(t_.value)
    barrier()

    # ---- the optional single-precision mode (north star: "held to 1e-4 relative and reported separately"): the same controller
    # instances and cycles with the fused kernel in FP32 (state, goals, integrators and torques stay FP64 in HBM), and its
    # error against the FP64 mode on a fresh pair of 4,096-robot batches (same states, same goals, 3 cycles each)
    fp32_ms, fp32_err = float("nan"), float("nan")
    if R >= 4096 and all(lib.osc_set_precision(s_["robot"].handle, capi.OSC_PRECISION_FP32) == 0 for s_ in sets):
        for s_ in sets:
            s_["robot"].setStream(stream.cuda_stream)     # the instances were on their own streams for the sections above
        torch.cuda.set_stream(stream)
        f_steps = max(args.steps, 100)
        for w in range(8):
            step_device(sets[w % n_sets])
        barrier()
        f_runs = []
        for _ in range(5):
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            f0.record()
            for k in range(f_steps):
                step_device(sets[k % n_sets])
            f1.record()
            barrier()
            f_runs.append(f0.elapsed_time(f1) / f_steps)
        fp32_ms = float(np.median(f_runs))
        fst = sets[0]["robot"].status()
        if (fst & capi.STATUS_UNHANDLED).any() or not bool(torch.isfinite(sets[0]["tau"]).all()) or \
                (args.min_ratio > 0 and (fst & capi.STATUS_SINGULAR_PATH).any()):
            raise SystemExit("bench: FP32 mode left the fused kernel or produced non-finite torques")
        for s_ in sets:
            lib.osc_set_precision(s_["robot"].handle, capi.OSC_PRECISION_FP64)
        pair = {}
        for mode in (capi.OSC_PRECISION_FP64, capi.OSC_PRECISION_FP32):
            probot = sp.BatchedRobot(ROBOT, 4096, device=local_rank)
            probot.setStream(stream.cuda_stream)
            probot.setQ(q[:4096]); probot.setDq(dq[:4096]); probot.updateModel()
            pm = sp.MotionForceTask(probot, LINK, (np.eye(3), np.array(POINT))); pj = sp.JointTask(probot)
            pm.disableInternalOtg(); pj.disableInternalOtg()
            pc = sp.RobotController(probot, [pm, pj])
            pm.setGoalPosition(goals["xd"][:4096]); pm.setGoalOrientation(goals["Rd"][:4096]); pm.setGoalLinearVelocity(goals["vd"][:4096])
            pm.setGoalAngularVelocity(goals["wd"][:4096]); pm.setGoalLinearAcceleration(goals["ad"][:4096]); pm.setGoalAngularAcceleration(goals["ald"][:4096])
            pj.setGoalPosition(goals["qd"][:4096])
            lib.osc_set_precision(probot.handle, mode)
            for _ in range(3):
                pc.updateControllerTaskModels()
                ptau = pc.computeControlTorques()
            pair[mode] = ptau
            del pc
            probot.close()
        ref64 = pair[capi.OSC_PRECISION_FP64]
        fp32_err = float((np.abs(pair[capi.OSC_PRECISION_FP32] - ref64).max(axis=1) / np.maximum(np.abs(ref64).max(axis=1), 1e-9)).max())
    barrier()

    # ---- max over ranks
    if world > 1:
        t = torch.tensor([e2e_ms, multi_ms, link_ms, unfiltered_ms, unfiltered_large_ms, fp32_ms, fp32_err], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms, multi_ms, link_ms, unfiltered_ms, unfiltered_large_ms, fp32_ms, fp32_err = (float(t[k]) for k in range(7))
    value = world * R * args.steps / (total_ms * 1e-3)
    e2e_value = world * R * e2e_steps / (e2e_ms * 1e-3)

    if rank == 0:
        # average duration of one cycle inside the timed region (fused kernel + the general-path kernel, which finds an
        # empty hand-over list on this workload): an upper bound of the fused kernel's own duration
        kernel_ms = total_ms / args.steps
        achieved_tflops = FLOP_PER_CYCLE * R / (kernel_ms * 1e-3) / 1e12
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        traffic = None      # dram__bytes_read.sum + dram__bytes_write.sum per launch, from the committed ncu --set full capture
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            if int(tr.get("robots", 0)) == R:
                traffic = {"bytes_per_launch": tr["dram_bytes_per_launch"], "source": tr["source"]}
        except Exception:
            pass
        bytes_per_cycle = 8 * (14 + 24 + 21 + 2 * 13 + 7 + 12)   # q,dq + goals + integrators r/w + tau + pose observers
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, world),
            "inputs": {"rejected_fraction": rejected, "robots_on_the_general_path": singular_fraction},
            "timing": {"timed_steps": args.steps, "timed_ms_total": total_ms, "setup_cycles": SETUP_ROUNDS * n_sets,
                       "warmup_cycles": args.warmup,
                       "what": "--steps back-to-back cycles after setup_cycles (every controller instance until its launch "
                               "configuration settles) and warmup_cycles, between two CUDA events with barrier + synchronize "
                               "on both sides; max over ranks"},
            "latency_ms": {"p50": float(np.percentile(per_step_ms, 50)), "p99": float(np.percentile(per_step_ms, 99)),
                           "max": float(per_step_ms.max()), "samples": int(per_step_ms.size), "what": "CUDA events around one batched cycle, rank 0"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(2 * n * R * 8), "d2h_bytes_per_step": int(n * R * 8),
                    "steps": e2e_steps, "passes_ms": [round(x, 3) for x in e2e_runs], "checksum": checksum,
                    "host_placement": placement,
                    "host_link": {"ms_per_step_copies_only": link_ms, "gbs": (3 * n * R * 8) / (link_ms * 1e-3) / 1e9,
                                  "e2e_fraction_of_link": link_ms / (e2e_ms / e2e_steps),
                                  "what": "the same %d + %d bytes per step as plain pinned cudaMemcpyAsync host->device and device->host on two "
                                          "streams at once, no kernel, max over ranks" % (2 * n * R * 8, n * R * 8)}},
            "extra": {"device_resident_one_stream_per_instance": {"value": world * R * multi_steps / (multi_ms * 1e-3), "unit": UNIT,
                      "what": "same cycles, the %d controller instances on their own streams (independent batches overlap), host clock" % n_sets},
                      "unfiltered_states": {"value": world * R / (unfiltered_ms * 1e-3), "unit": UNIT, "ms_per_step": unfiltered_ms,
                                            "robots_on_the_general_path": unfiltered_singular,
                                            "what": "same hierarchy and batch size, uniformly sampled states without the s_min/s_max filter: the "
                                                    "robots inside the reference's blending band take the general (SVD) path; 30 cycles, CUDA events"},
                      "fp32_mode": (None if not (fp32_ms == fp32_ms) else
                                    {"value": world * R / (fp32_ms * 1e-3), "unit": UNIT, "ms_per_step": fp32_ms, "dtype": "f32",
                                     "max_relative_error_vs_fp64": fp32_err, "tolerance": 1e-4,
                                     "fraction_of_fp32_roofline": FLOP_PER_CYCLE * R / (fp32_ms * 1e-3) / 1e12 / FP32_PEAK_TFLOPS,
                                     "what": "optional single-precision mode (osc_set_precision): the same instances and cycles with the fused kernel in FP32 "
                                             "arithmetic on FP64 state; reported separately, not part of `value`; the error is per robot, "
                                             "max |tau32 - tau64| / max |tau64|, 4,096 robots, third cycle; roofline against %.1f TFLOP/s FP32 "
                                             "(148 SM x 128 FMA/clk x 2 x 1.965 GHz)" % FP32_PEAK_TFLOPS}),
                      "unfiltered_states_1m_robots": (None if not (unfiltered_large_ms == unfiltered_large_ms) else
                                                      {"value": world * R_LARGE / (unfiltered_large_ms * 1e-3), "unit": UNIT, "ms_per_step": unfiltered_large_ms,
                                                       "robots_per_gpu": R_LARGE, "robots_on_the_general_path": unfiltered_large_singular,
                                                       "what": "the same at 1,048,576 robots per GPU: the hand-over list is many waves long and takes the split "
                                                               "blending path (classification kernel, one variant per warp); 10 cycles, CUDA events"})},
            "gpu_launches": int(launches),
            "clocks": clk,
            "roofline": {"bound": "fp64", "achieved": achieved_tflops, "peak": FP64_PEAK_TFLOPS, "unit": "TFLOP/s",
                         "frac": achieved_tflops / FP64_PEAK_TFLOPS, "traffic": traffic,
                         "kernel": "osc_cycle_kernel<7,6,JT,FULL,SPEC>", "kernel_ms": kernel_ms,
                         "flop_per_robot_cycle": FLOP_PER_CYCLE,
                         "fp64_measured": {"tflops": fp64_measured, "frac": (achieved_tflops / fp64_measured) if fp64_measured else None,
                                           "how": "DFMA-only kernel, 8 chains per thread, 64 warps per SM, best launch of the second half of 0.4 s (osc_measure_fp64_peak)"},
                         "peak_source": "datasheet-derived FP64 FMA peak (148 SM x 64 FMA/clk x 2 x 1.965 GHz); MEASURED_PEAKS.json has no FP64 entry",
                         "hbm": {"achieved_gbs": bytes_per_cycle * R / (kernel_ms * 1e-3) / 1e9, "peak_gbs": hbm_peak,
                                 "bytes_per_robot_cycle": bytes_per_cycle, "peak_source": "of measured" if peaks else "of fallback"}},
        }
        # CPU baseline on rank 0 at N=1 only
        if world == 1 and not args.no_cpu:
            n_sample = min(R, 16384)
            res = run_cpu_baseline(n_sample, args.cpu_seconds, q, dq, goals)
            kind = "reference" if "reference" in res else "port"
            v, med, reps, threads = res[kind]
            out["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": kind,
                                   "sample": "%d robots of the same batch x 1 cycle, median of %d runs (%.3f s each), %s, incl. the model update, "
                                             "%d host threads" % (n_sample, reps, med, KIND_TEXT[kind], threads)}
            if kind == "reference":
                out["cpu_baseline"]["port"] = {"value": res["port"][0], "what": KIND_TEXT["port"] + ", same sample and threads"}
        else:
            out["cpu_baseline"] = None
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--robots", type=int, default=65536, help="robots per GPU (BASELINE config 2: 65,536)")
    ap.add_argument("--sets", type=int, default=8, help="controller instances used round-robin (working set > L2)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-seconds", type=float, default=16.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--min-ratio", type=float, default=0.1, help="reject states with s_min/s_max below this (0: unfiltered, about half of the Panda states then take the singular branch)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the torques of the last timed cycle to DIR/tau.npy (float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        reference_arm(args)
    else:
        gpu_arm(args)


if __name__ == "__main__":
    main()
