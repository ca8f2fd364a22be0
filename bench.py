#!/usr/bin/env python
"""bench.py — BASELINE.json metric: QP solves/sec (N=12, nx=6, nu=2).

Headline workload = BASELINE.json configs[1]: batch=4096 LTV-MPC QPs, N=12, per-instance fixed (A_k,B_k,C_k)
(126 variables / 174 constraint rows each in the reference's OSQP form), built by racinglmpc_b200/workloads.py from the
committed fixture (SURVEY §8d).  One "step" = one pass of the hot path (assemble-free QP solve + unpack, one kernel launch)
over the whole batch.  The same line carries, under "configs", the other BASELINE configurations measured in the same
process so that the driver's records cover them:
  configs[2]  batch=4096 full LMPC steps (k-NN regression K1 -> safe-set selection K2 -> 180-variable QP -> shift), with
              per-kernel durations and rooflines (K1 against HBM, the QP kernels against the measured fp64 peak);
  configs[3]  LMPC Monte-Carlo rollouts, 8192 controllers per GPU, device-resident closed loop, pooled safe-set exchange with
              one NCCL all-gather per lap (benchmarks/rollout_mc.py).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config 1|2|3] [--dump-outputs DIR]

`--dump-outputs DIR` writes, after the timed steps, what the last timed step of configs[1] and configs[2] returned to its caller
as DIR/config1_<name>.npy and DIR/config2_<name>.npy (float64; inputs are seeded, so two builds can be compared array by array).

Under torchrun (N > 1) every rank owns its own batch on its own GPU (weak scaling; instances are independent — SURVEY §8e);
timing is CUDA events on the launching stream, max over ranks.  `--impl reference` times the CPU oracle
(oracle/osqp_port.c: the OSQP algorithm with the reference's settings, cold start + polish, PC.py:259-283) on the host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True      # the tree may be read-only; nothing of a run is written into it

# one OpenMP thread per physical core, pinned: the CPU arm has to be repeatable (set before the oracle library loads)
os.environ.setdefault("OMP_PROC_BIND", "spread")
os.environ.setdefault("OMP_PLACES", "cores")

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "QP solves/sec (N=12, nx=6, nu=2)"
UNIT = "solves/s"
BATCH = 4096
HORIZON = 12
WORKLOAD = "configs[1]: batch=4096 LTV-MPC QPs N=12 nx=6 nu=2, per-instance fixed A/B/C (126 vars / 174 rows in OSQP form)"
CPU_SAMPLE = 1024          # QPs of the workload the CPU arm solves per step (bounded sample, both arms)
# algorithmic HBM bytes per solve (SURVEY §8d, config 2, per-instance A/B/C):
#   in  x0 6 + OldInput 2 + ABC 648 = 656 f64 ; out xPred 78 + uPred 24 + status/iters/3 resid ~4 = 106 f64
ALGO_BYTES_PER_SOLVE = (656 + 106) * 8
SS_BYTES_PER_SOLVE = (6 * 48 + 48 + 6 * 48 + 2 * 48) * 8           # selected safe set + successors read by the LMPC QP
# algorithmic fp64 flops of one interior-point iteration (N = 12; DESIGN.md §4): Riccati factorisation 12 stages x
# (A~'PA~ 2*8*8*8*... counted on the 6x8 / 8x8 blocks actually needed) + three vector sweeps + row updates
FLOPS_PER_ITER = 12 * 2 * (288 + 216 + 126 + 72 + 36 + 48) + 4 * 12 * 2 * 126 + 4000
FLOPS_PER_ITER_LMPC = FLOPS_PER_ITER + 2 * 48 * (21 + 6 * 6) + 2000       # + simplex terminal block (W assembly, recoveries)
# fp64 tensor-core instructions issued per iteration: 12 stages x (11 factor + 4 corrector gradient + 2 x 4 forward)
DMMA_PER_ITER = 12 * (11 + 4 + 8) + 2 * 6 + 2 * 2     # sweeps per stage + stage-gradient / right-hand-side tiles of 8 stages
DUMP_LIMIT = 60 * 10**6          # array bytes --dump-outputs writes at most: below 64 MB with the .npy headers


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 9:
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------
# CPU oracle arm (cpu_baseline leg and --impl reference).  The ONLY place bench.py touches oracle/.
# ----------------------------------------------------------------------------------------------
def oracle_problem_set(nsample, seed=1):
    """Assemble `nsample` of the workload's QPs in the reference's OSQP form (Python, untimed)."""
    from oracle import ftocp, osqp_port
    from racinglmpc_b200 import workloads
    x0, uold, abc = workloads.ltv_mpc_batch(nsample, N=HORIZON, seed=seed)
    par = ftocp.mpc_params(6, 2, HORIZON, 0.8)[1]
    par.timeVarying = True
    F, bb = ftocp.build_ineq(par)
    Ps, qs, As, ls, us = [], [], [], [], []
    for b in range(nsample):
        A = abc[b][:, 0:36].reshape(HORIZON, 6, 6)
        Bm = abc[b][:, 36:48].reshape(HORIZON, 6, 2)
        C = abc[b][:, 48:54]
        H, q = ftocp.build_cost(par, uold[b])
        G, E, L = ftocp.build_eq(par, list(A), list(Bm), list(C))
        P, q, Am, l, u = ftocp.osqp_form(H, q, F, bb, G, E @ x0[b] + L)
        Ps.append(P); qs.append(q); As.append(Am); ls.append(l); us.append(u)
    maskP = np.any(np.array([p != 0 for p in Ps]), axis=0)
    maskA = np.any(np.array([a != 0 for a in As]), axis=0)
    patP, patA = osqp_port.csc_pattern(maskP, maskA)
    Px = np.stack([osqp_port.gather_values(p, *patP) for p in Ps])
    Ax = np.stack([osqp_port.gather_values(a, *patA) for a in As])
    return patP, patA, Px, np.stack(qs), Ax, np.stack(ls), np.stack(us)


def oracle_pass(prob, nthreads):
    """One pass of the CPU arm over the sample: (seconds, solved, mean ADMM iterations)."""
    from oracle import osqp_port
    patP, patA, Px, q, Ax, l, u = prob
    t0 = time.perf_counter()
    _, infos, _ = osqp_port.solve_batch(patP, patA, Px, q, Ax, l, u, nthreads=nthreads)
    dt = time.perf_counter() - t0
    return dt, sum(1 for i in infos if i["status"] == 1), float(np.mean([i["iters"] for i in infos]))


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


_CPU_THREADS = None


def cpu_threads():
    """Cached: the affinity mask must be read BEFORE the OpenMP runtime of the oracle library loads (with OMP_PROC_BIND set it
    pins the calling thread to one core, after which sched_getaffinity reports a single CPU)."""
    global _CPU_THREADS
    if _CPU_THREADS is None:
        _CPU_THREADS = _cpu_threads()
    return _CPU_THREADS


def _cpu_threads():
    """Threads of the CPU arm, fixed by the machine instead of searched: one per PHYSICAL core of the affinity mask, capped by the
    container's CPU quota (SMT siblings slow this solver down: measured 16 k solves/s on 128 hardware threads against 150-175 k on
    the 64 cores behind them).  LMPC_BENCH_THREADS overrides.  Returns (threads, description)."""
    if os.environ.get("LMPC_BENCH_THREADS"):
        n = max(1, int(os.environ["LMPC_BENCH_THREADS"]))
        return n, "LMPC_BENCH_THREADS=%d" % n
    try:
        cpus = sorted(os.sched_getaffinity(0))
    except AttributeError:
        cpus = list(range(os.cpu_count() or 1))
    cores = set()
    for c in cpus:
        try:
            pkg = open("/sys/devices/system/cpu/cpu%d/topology/physical_package_id" % c).read().strip()
            cid = open("/sys/devices/system/cpu/cpu%d/topology/core_id" % c).read().strip()
            cores.add((pkg, cid))
        except OSError:
            cores.add(("?", c))
    phys = max(1, len(cores))
    quota = None
    try:                                                    # cgroup v2, then v1
        qs, ps = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if qs != "max":
            quota = max(1, int(int(qs) // int(ps)))
    except (OSError, ValueError):
        try:
            qv = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            pv = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if qv > 0:
                quota = max(1, qv // pv)
        except (OSError, ValueError):
            pass
    n = min(phys, quota) if quota else phys
    return n, "%d physical cores of %d logical CPUs%s" % (phys, len(cpus), (", CPU quota %d" % quota) if quota else "")


def cpu_arm(prob, repeats=5):
    """The CPU arm, identical for `--impl reference` and the GPU arm's cpu_baseline leg: fixed thread count, one untimed pass,
    `repeats` timed passes, median.  Returns a dict."""
    n, how = cpu_threads()
    nsample = prob[3].shape[0]
    oracle_pass(prob, n)
    ts, solved, iters = [], 0, 0.0
    for _ in range(repeats):
        dt, s, it = oracle_pass(prob, n)
        ts.append(dt); solved = s; iters = it
    med = float(np.median(ts))
    return {"value": nsample / med, "threads": n, "threads_how": how, "per_thread": nsample / med / n, "passes_s": [round(t, 4) for t in ts],
            "spread": (max(ts) - min(ts)) / med, "solved_fraction": solved / nsample, "mean_admm_iters": iters}


def cpu_baseline_block(arm):
    return {"value": arm["value"], "unit": UNIT, "cores": arm["threads"], "kind": "port",
            "sample": "first %d of the 4096 QPs per pass, OSQP-algorithm C port with the reference's settings (eps 1e-3, polish, cold start "
                      "per QP; PC.py:259-283), median of %d passes on %s (pass-to-pass spread %.1f %%), %.0f solves/s per thread; cpu %s"
                      % (CPU_SAMPLE, len(arm["passes_s"]), arm["threads_how"], 100 * arm["spread"], arm["per_thread"], cpu_model())}


def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return
    prob = oracle_problem_set(CPU_SAMPLE)
    n, _ = cpu_threads()
    for _ in range(args.warmup):
        oracle_pass(prob, n)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        oracle_pass(prob, n)
    dt = time.perf_counter() - t0
    arm = cpu_arm(prob)
    val = CPU_SAMPLE * args.steps / dt
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample_per_step": CPU_SAMPLE, "cpu": cpu_model(), "solved_fraction": arm["solved_fraction"],
                   "mean_admm_iters": arm["mean_admm_iters"], "median_of_5_passes": arm["value"]},
        "cpu_baseline": dict(cpu_baseline_block(arm), value=val),
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


# ----------------------------------------------------------------------------------------------
# GPU legs
# ----------------------------------------------------------------------------------------------
def _peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def _traffic(kernel):
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[kernel]["dram_bytes_per_launch"]
    except Exception:
        return None


def dump_outputs(path, groups):
    """--dump-outputs: every array of ``groups`` ({prefix: {name: array[B, ...]}}) as path/<prefix>_<name>.npy in float64.  Above
    DUMP_LIMIT bytes in all, each group keeps the same fixed, seeded sample of its B instances (indices in <prefix>_sample_index.npy)."""
    row_bytes = {p: 8 * (1 + sum(np.asarray(a)[0].size for a in g.values())) for p, g in groups.items()}
    total = sum(row_bytes[p] * len(next(iter(g.values()))) for p, g in groups.items())
    frac = min(1.0, DUMP_LIMIT / total)
    os.makedirs(path, exist_ok=True)
    for p, g in groups.items():
        B = len(next(iter(g.values())))
        idx = np.arange(B)
        if frac < 1.0:
            idx = np.sort(np.random.default_rng(0).choice(B, max(1, int(B * frac)), replace=False))
            np.save(os.path.join(path, p + "_sample_index.npy"), idx.astype(np.float64))
        for name, a in g.items():
            np.save(os.path.join(path, "%s_%s.npy" % (p, name)), np.asarray(a)[idx].astype(np.float64))


def _max_over_ranks(v, dev, world):
    import torch
    import torch.distributed as dist
    t = torch.tensor([float(v)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def _pinner(local):
    """Host buffers of the end-to-end legs: the library's pinned allocator (lmpc_host_alloc); if the host refuses to register
    memory (locked-memory limit), torch's pinned allocator -- still pinned, only slower for a single DMA stream."""
    import torch
    from racinglmpc_b200 import _native as nat

    def pin(a):
        a = np.ascontiguousarray(a)
        try:
            return nat.pinned_like(a, device=local)
        except nat.NativeError as e:
            print("bench: lmpc_host_alloc failed (%s); using torch pinned memory" % e, file=sys.stderr)
            return torch.from_numpy(a).pin_memory().numpy()
    return pin


def leg_config1(args, rank, world, local, dev):
    """configs[1]: device-timed value + end-to-end through the public host API."""
    import torch
    import torch.distributed as dist
    from racinglmpc_b200 import BatchedFTOCP, workloads, reference_params as rp
    B, N = BATCH, HORIZON
    x0, uold, abc = workloads.ltv_mpc_batch(B, N=N, seed=1 + rank)
    solver = BatchedFTOCP(rp.mpc_params(N), batch=B, device=local)
    stream = torch.cuda.ExternalStream(solver.stream, device=dev)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    d_x0, d_u, d_abc = t(x0), t(uold), t(abc)
    d_xP = torch.zeros(B, N + 1, 6, dtype=torch.float64, device=dev)
    d_uP = torch.zeros(B, N, 2, dtype=torch.float64, device=dev)
    d_st = torch.zeros(B, dtype=torch.int32, device=dev)
    d_it = torch.zeros(B, dtype=torch.int32, device=dev)
    d_rs = torch.zeros(B, 3, dtype=torch.float64, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2
    torch.cuda.synchronize()

    def step_dev():
        solver.solve_dev(d_x0, d_u, d_abc, N * 54, 54, d_xP, d_uP, d_st, d_it, d_rs)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()            # runs through warm-up and the device-timed region (under load)
    for _ in range(max(args.warmup, 3)):
        step_dev()
    solver.sync()
    t_w = time.perf_counter()      # extra untimed warm-up: >= 0.4 s of load so that clocks settle and get sampled
    while time.perf_counter() - t_w < 0.4:
        for _ in range(8):
            step_dev()
        solver.sync()
    launches0 = solver.kernel_launches
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    with torch.cuda.stream(stream):
        for i in range(args.steps):
            flush.zero_()                      # L2 flush between timed iterations (same stream, untimed)
            ev[i][0].record(stream)
            step_dev()
            ev[i][1].record(stream)
    solver.sync()
    barrier()
    launches = solver.kernel_launches - launches0
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = _max_over_ranks(sum(step_ms), dev, world)
    status, iters, resid = d_st.cpu().numpy(), d_it.cpu().numpy(), d_rs.cpu().numpy()
    outputs = None
    if args.dump_outputs:
        outputs = dict(xPred=d_xP.cpu().numpy(), uPred=d_uP.cpu().numpy(), status=status, iters=iters, resid=resid)
    # nvidia-smi polling takes driver locks that stall cudaMemcpyAsync enqueues: the sampler covers the device-timed region
    # only and is stopped before the host-timed leg (measured: 2.6-3.4 M/s with it running, 3.9 M/s without)
    clocks = sampler.stop() if rank == 0 else None

    # ---- end-to-end: the public host API, used the way a caller streams batch after batch: three batches in flight (solve_async on
    # rotating buffer sets, wait before a set is reused), pinned host buffers; every step's inputs are copied H2D and every step's results
    # D2H inside the timed region
    # pinned host buffers from the library's allocator: pages on the NUMA node of the GPU's PCIe link (lmpc_host_alloc)
    from racinglmpc_b200 import _native as nat
    pin = _pinner(local)
    h_x0, h_u, h_abc = pin(x0), pin(uold), pin(abc)
    nslot = max(1, min(4, int(os.environ.get("LMPC_B200_E2E_SLOTS", "3"))))   # batches in flight (measurement knob)
    outs = [{k: pin(v) for k, v in solver.alloc_outputs(False).items()} for _ in range(nslot)]
    for i in range(max(args.warmup, 3) + 20):   # untimed; long enough to bring the clocks back up after the pinning pause
        slot = i % nslot
        if i >= nslot:
            solver.wait(slot)
        solver.solve_async(slot, h_x0, h_u, h_abc, outs[slot])
    for sl in range(nslot):
        solver.wait(sl)
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        slot = i % nslot
        if i >= nslot:
            solver.wait(slot)                  # results of step i-nslot are on the host before its buffer set is reused
        solver.solve_async(slot, h_x0, h_u, h_abc, outs[slot])
    for sl in range(nslot):
        solver.wait(sl)
    torch.cuda.synchronize()
    out = outs[(args.steps - 1) % nslot]
    e2e_s = _max_over_ranks(time.perf_counter() - t0, dev, world)
    late = solver.late_accepts
    solver.close()
    return dict(B=B, total_ms=total_ms, step_ms=step_ms, launches=int(launches), status=status, iters=iters, resid=resid, clocks=clocks,
                e2e_s=e2e_s, h2d=int(h_x0.nbytes + h_u.nbytes + h_abc.nbytes),
                d2h=int(sum(out[k].nbytes for k in ("xPred", "uPred", "slack", "status", "iters", "resid"))), late=late, outputs=outputs)


def leg_config2(args, rank, world, local, dev, with_e2e=True):
    """configs[2]: full LMPC steps (K1 -> K2 -> QP<12,48> -> shift), per-instance 5-lap stores."""
    import torch
    import torch.distributed as dist
    from racinglmpc_b200 import workloads, reference_params as rp
    from racinglmpc_b200.controller import BatchedController
    B, N = args.batch, HORIZON
    steps = args.steps
    seg = workloads.track_seg_table()      # Map.PointAndTangent[:,3:6] from the reference-pinned fixture
    data = workloads.lmpc_batch(B, seed=2 + rank)
    numSS_it, numSS_Points, _, _, Qts, par = rp.lmpc_params(N)
    c = BatchedController(par, B, seg, rp.TRACK_LENGTH, trToUse=5, numSS_Points=numSS_Points, numSS_it=numSS_it,
                          QterminalSlack=Qts, device=local, Tmax=1280, ss_cap=5, model_cap=5)
    workloads.restore_lmpc_batch(c, data)
    stream = torch.cuda.ExternalStream(c.stream, device=dev)
    d_x0 = torch.from_numpy(data["x0"]).to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    state = dict(xLin=data["xLin"], uLin=data["uLin"], zt=data["zt"], OldInput=data["OldInput"],
                 timeStep=data["t"].astype(np.int32), has_pred=np.ones(B, np.int32), xPred=data["xPred"])

    def reset():
        c.set_state(**state)      # every timed step solves the same controller states (untimed host upload)

    for _ in range(max(args.warmup, 3)):
        reset(); c.step_dev(d_x0); c.sync()
    l0 = c.kernel_launches
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    for i in range(steps):
        reset()
        with torch.cuda.stream(stream):
            flush.zero_()
            ev[i][0].record(stream)
            c.step_dev(d_x0)
            ev[i][1].record(stream)
        c.sync()
    launches = c.kernel_launches - l0
    torch.cuda.synchronize()
    # the device-resident step hands its caller the step results and the shifted controller state
    outputs = dict(c.step_results(), **c.get_state()) if args.dump_outputs else None
    step_ms = [a.elapsed_time(b) for a, b in ev]
    tot = _max_over_ranks(sum(step_ms), dev, world)
    # per-kernel durations (CUDA events between the four launches of one step, L2 flushed, median of a few steps)
    kms = []
    for _ in range(5):
        reset()
        with torch.cuda.stream(stream):
            flush.zero_()
        c.sync()
        kms.append(c.step_profile(d_x0))
    kms = np.median(np.array(kms), axis=0)
    res = c.step_results()
    ok = float(np.mean((res["status"] == 1) & (res["flags"] == 0)))
    e2e = None
    if with_e2e:       # host x0 in, results out through the public API
        from racinglmpc_b200 import _native as nat
        pin = _pinner(local)
        h_x0 = pin(data["x0"])
        out = {k: pin(v) for k, v in c.alloc_step_outputs().items()}
        reset(); c.step(h_x0, out=out, want_ss=False)
        t_e2e = 0.0
        for _ in range(steps):
            reset()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            c.step(h_x0, out=out, want_ss=False)
            t_e2e += time.perf_counter() - t0
        e2e = {"value": B * world * steps / _max_over_ranks(t_e2e, dev, world), "unit": UNIT, "h2d_bytes_per_step": int(h_x0.nbytes),
               "d2h_bytes_per_step": int(sum(out[k].nbytes for k in ("xPred", "uPred", "lambd", "zt", "zt_u", "status", "iters", "resid", "flags")))}
    rows_model = sum(l[0].shape[0] for l in data["model_laps"][0])
    rows_ss = sum(l[0].shape[0] for l in data["ss_laps"][0])
    late = c.late_accepts
    c.close()
    return dict(B=B, steps=steps, total_ms=tot, launches=int(launches), kernel_ms=[float(v) for v in kms], ok=ok, iters=res["iters"],
                rows_model=rows_model, rows_ss=rows_ss, e2e=e2e, data=data, late=late, outputs=outputs)


def config2_block(r, world, probe, peaks):
    """JSON block of the configs[2] leg with per-kernel rooflines."""
    B = r["B"]
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    k1, k2, qp, sh = r["kernel_ms"]
    k1_bytes = B * r["rows_model"] * 64.0                      # one pass over the used laps: x (48 B) + u (16 B) per stored row
    k2_bytes = B * r["rows_ss"] * 48.0                         # one pass over the states of the numSS_it fastest laps
    flops = float(np.sum(r["iters"] + 1)) * FLOPS_PER_ITER_LMPC
    qp_tf = flops / (qp * 1e-3) / 1e12
    ms = r["total_ms"] / r["steps"]
    algo = r["rows_model"] * 64 + r["rows_ss"] * 48 + ALGO_BYTES_PER_SOLVE + SS_BYTES_PER_SOLVE
    return {"workload": "configs[2]: batch=%d full LMPC steps (k-NN LTV regression over a 5-lap store, 4-lap sampled safe set, 180 vars / 229 "
                        "rows QP), N=12" % B,
            "value": B * world * r["steps"] / (r["total_ms"] * 1e-3), "unit": "controller steps/s", "ms_per_step": ms, "steps": r["steps"],
            "gpu_launches": r["launches"], "solved_fraction": r["ok"], "ipm_iters_mean": float(r["iters"].mean()),
            "ipm_iters_max": int(r["iters"].max()), "late_accepts": r["late"], "e2e": r["e2e"],
            "kernels": {
                "knn_ltv_regress_kernel": {"ms": k1, "roofline": {"bound": "hbm", "achieved": k1_bytes / (k1 * 1e-3) / 1e9, "peak": hbm_peak,
                                                                  "unit": "GB/s", "frac": k1_bytes / (k1 * 1e-3) / 1e9 / hbm_peak,
                                                                  "traffic": _traffic("knn_ltv_regress_kernel"),
                                                                  "algorithmic_bytes_per_launch": k1_bytes}},
                "ss_select_kernel": {"ms": k2, "roofline": {"bound": "hbm", "achieved": k2_bytes / (k2 * 1e-3) / 1e9, "peak": hbm_peak,
                                                            "unit": "GB/s", "frac": k2_bytes / (k2 * 1e-3) / 1e9 / hbm_peak, "traffic": None}},
                "ftocp_kernel<12,48,2,4>": {"ms": qp, "roofline": {"bound": "tensor", "achieved": qp_tf, "peak": probe["dmma_tflops"],
                                                                   "unit": "TFLOP/s", "frac": qp_tf / probe["dmma_tflops"],
                                                                   "traffic": _traffic("ftocp_kernel<12,48,2,4>"),
                                                                   "peak_source": "measured on this GPU (lmpc_probe_fp64: mma.sync.m8n8k4.f64)"}},
                "shift_state_kernel": {"ms": sh}},
            "whole_step_hbm": {"algorithmic_bytes_per_step": algo, "achieved_gbs": B * algo / (ms * 1e-3) / 1e9}}


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from racinglmpc_b200 import _native

    rank, world, local = dist_env()
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    peaks = _peaks()
    probe = _native.probe_fp64(local)              # measured fp64 numbers of THIS GPU: the QP kernels' roofline denominators

    r1 = leg_config1(args, rank, world, local, dev)
    B, iters = r1["B"], r1["iters"]
    line = None
    if rank == 0:
        value = B * world * args.steps / (r1["total_ms"] * 1e-3)
        kern_ms = float(np.mean(r1["step_ms"]))                 # one kernel per step: launch duration == step duration
        tflops = float(np.sum(iters + 1)) * FLOPS_PER_ITER / (kern_ms * 1e-3) / 1e12
        issued = float(np.sum(iters + 1)) * DMMA_PER_ITER * 512 / (kern_ms * 1e-3) / 1e12
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        hbm_ach = B * ALGO_BYTES_PER_SOLVE / (kern_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": r1["total_ms"] / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_gpu": B, "horizon": HORIZON,
                       "l2": "flushed between timed steps (256 MiB memset on the same stream)",
                       "e2e_mode": "public host API with three batches in flight (solve_async/wait on rotating buffer sets), pinned host "
                                   "buffers from lmpc_host_alloc (pages on the GPU's NUMA node); every step copies its inputs H2D and its results D2H "
                                   "inside the timed region",
                       "host_numa_node": int(_native.lib().lmpc_host_numa_node(local)),
                       "tolerance": "r_prim, r_dual <= 1e-9, gap <= 1e-11 (unscaled inf-norm), last primal step <= 1e-7",
                       "solved_fraction": float(np.mean(r1["status"] == 1)), "ipm_iters_mean": float(iters.mean()),
                       "ipm_iters_max": int(iters.max()), "max_resid": float(r1["resid"].max()), "late_accepts": r1["late"]},
            "clocks": r1["clocks"],
            "e2e": {"value": B * world * args.steps / r1["e2e_s"], "unit": UNIT, "h2d_bytes_per_step": r1["h2d"], "d2h_bytes_per_step": r1["d2h"]},
            "gpu_launches": r1["launches"],
            "roofline": {"bound": "tensor", "achieved": tflops, "peak": probe["dmma_tflops"], "unit": "TFLOP/s", "frac": tflops / probe["dmma_tflops"],
                         "traffic": _traffic("ftocp_kernel<12,0,2,4>"), "kernel": "ftocp_kernel<12,0,2,4>",
                         "peak_source": "measured on this GPU by lmpc_probe_fp64 (mma.sync.m8n8k4.f64, the instruction the Riccati sweeps issue); "
                                        "MEASURED_PEAKS.json holds no fp64 number",
                         "note": "achieved = algorithmic fp64 flops of the interior-point iterations / kernel time; the tensor-core instructions "
                                 "actually issued (8x8x4 fragments, row vectors padded to 8 rows) are `issued_tflops`",
                         "issued_tflops": issued, "issued_frac": issued / probe["dmma_tflops"], "fp64_probe": probe,
                         "hbm": {"achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_ach / hbm_peak,
                                 "algorithmic_bytes_per_solve": ALGO_BYTES_PER_SOLVE,
                                 "peak_source": "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"}},
        }
    dumps = {"config1": r1["outputs"]}
    # ---- the other BASELINE configurations, same process, all ranks (weak scaling: every rank its own batch)
    if not args.headline_only:
        r2 = leg_config2(args, rank, world, local, dev)
        dumps["config2"] = r2["outputs"]
        from benchmarks import rollout_mc
        r3 = rollout_mc.run(batch=args.rollout_batch, laps=3, mode="pooled", share=2, local=local)
        if rank == 0:
            r3["workload"] = ("configs[3]: LMPC Monte-Carlo rollouts, %d controllers per GPU x %d GPUs, device-resident closed loop (main.py's "
                              "PID lap -> seeding -> 3 LMPC laps), pooled safe-set exchange: one NCCL all-gather per lap" % (args.rollout_batch, world))
            line["configs"] = {"configs[2]": config2_block(r2, world, probe, peaks), "configs[3]": r3}
    if rank == 0:
        if not args.no_cpu_baseline and world == 1:       # the CPU leg is measured at N = 1 only (rank 0 has the host to itself)
            line["cpu_baseline"] = cpu_baseline_block(cpu_arm(oracle_problem_set(CPU_SAMPLE)))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dumps)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_lmpc_steps(args):
    """--config 2 as its own line."""
    import torch
    import torch.distributed as dist
    from racinglmpc_b200 import _native
    rank, world, local = dist_env()
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    r = leg_config2(args, rank, world, local, dev)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        blk = config2_block(r, world, _native.probe_fp64(local), _peaks())
        ms = blk["ms_per_step"]
        line = {"metric": METRIC, "value": blk["value"], "unit": UNIT, "n_gpus": world, "steps": r["steps"], "warmup": max(args.warmup, 3),
                "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": blk["workload"], "batch_per_gpu": r["B"], "l2": "flushed between timed steps (256 MiB memset on the same stream)",
                           "solved_fraction": r["ok"], "ipm_iters_mean": blk["ipm_iters_mean"], "ipm_iters_max": blk["ipm_iters_max"],
                           "kernels_per_step": "knn_ltv_regress, ss_select, ftocp_kernel<12,48>, shift_state"},
                "clocks": clocks, "e2e": blk["e2e"], "gpu_launches": r["launches"], "kernels": blk["kernels"],
                "roofline": dict(blk["kernels"]["ftocp_kernel<12,48,2,4>"]["roofline"], kernel="ftocp_kernel<12,48,2,4>")}
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = lmpc_cpu_baseline(r["data"])
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"config2": r["outputs"]})
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_rollouts(args):
    """--config 3 as its own line."""
    import torch
    import torch.distributed as dist
    from benchmarks import rollout_mc
    rank, world, local = dist_env()
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    r = rollout_mc.run(batch=args.rollout_batch, laps=3, mode="pooled", share=2, local=local)
    if rank == 0:
        print(json.dumps({"metric": "LMPC closed-loop controller steps/sec (configs[3])", "value": r["controller_steps_per_s"], "unit": "steps/s",
                          "n_gpus": world, "steps": r["closed_loop_steps"], "warmup": 0, "ms_per_step": r["ms_total"] / r["closed_loop_steps"],
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                          "config": {"workload": "configs[3]: LMPC Monte-Carlo rollouts, %d controllers per GPU, pooled safe-set exchange"
                                                 % args.rollout_batch}, "detail": r}))
    if world > 1:
        dist.destroy_process_group()


def lmpc_cpu_baseline(data, nsample=24):
    """The reference's own way: one Python controller, one QP at a time (PC.py:110-137), restated by the oracle and
    solved by the OSQP-algorithm port with the reference's settings."""
    from oracle import ftocp, ltv_model, osqp_port
    from oracle.track import TrackTable
    trk = TrackTable()
    numSS_it, numSS_Points, _, _, Qts, par = ftocp.lmpc_params(trk, HORIZON)
    par.timeVarying = True
    ctrls = []
    for b in range(nsample):
        pm = ltv_model.LocalLTVModel(6, 2, trk, 5)
        pm.xStored = [lx for lx, _ in data["model_laps"][b]]
        pm.uStored = [lu for _, lu in data["model_laps"][b]]
        pm.lapTime = [lx.shape[0] for lx in pm.xStored]
        lm = ftocp.OracleLMPC(numSS_Points, numSS_it, Qts, par, pm, qp=osqp_port.reference_qp)
        lm.SS = [s[0] for s in data["ss_laps"][b]]; lm.uSS = [s[1] for s in data["ss_laps"][b]]
        lm.Qfun = [s[2] for s in data["ss_laps"][b]]; lm.LapTime = list(data["lap_times"])
        lm.it, lm.timeStep = 4, int(data["t"][b])
        lm.zt, lm.xLin, lm.uLin = data["zt"][b].copy(), data["xLin"][b].copy(), data["uLin"][b].copy()
        lm.OldInput, lm.xPred = data["OldInput"][b].copy(), data["xPred"][b].copy()
        ctrls.append(lm)
    t0 = time.perf_counter()
    for b, lm in enumerate(ctrls):
        lm.solve(data["x0"][b])
    dt = time.perf_counter() - t0
    return {"value": nsample / dt, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": "%d controller steps, oracle restatement of LMPC.solve in Python (as the reference: single thread) + "
                      "OSQP-algorithm C port, reference settings; cpu %s" % (nsample, cpu_model())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU oracle leg (profiling runs)")
    ap.add_argument("--headline-only", action="store_true", help="configs[1] only: skip the configs[2] / configs[3] legs (profiling runs)")
    ap.add_argument("--config", type=int, default=0, choices=[0, 1, 2, 3],
                    help="0 (default) = the headline line: configs[1] as `value`, configs[2] and configs[3] under `configs`; "
                         "1 = configs[1] only; 2 = batch=4096 full LMPC steps as its own line; 3 = Monte-Carlo rollouts as its own line")
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--rollout-batch", type=int, default=8192, help="controllers per GPU of the configs[3] leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step of configs[1] / configs[2] returned as DIR/*.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.config == 3):
        ap.error("--dump-outputs covers the configs[1] and configs[2] legs of the GPU implementation")
    cpu_threads()                 # read the affinity mask before any OpenMP runtime pins this thread
    if args.config == 1:
        args.headline_only = True
    if args.impl == "reference":
        run_reference(args)
    elif args.config == 2:
        run_lmpc_steps(args)
    elif args.config == 3:
        run_rollouts(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
