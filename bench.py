#!/usr/bin/env python
"""Benchmark of the hot path: converged trajectories / second of the batched trust-region SQP
(BASELINE.json metric), one process per GPU.

  python bench.py --gpus N --steps K --warmup W        # CUDA path (this repo)
  python bench.py --impl reference ...                  # CPU arm: the oracle restatement of the reference's CPU
                                                        # path on the host cores, SAME batches (seeds) as the CUDA arm

A "step" = one complete tb200_solve_batch over one batch of synthetic problems.  Default workload: 1024 x 7-DOF x 30
waypoints with the 8-sphere discrete collision constraint (BASELINE.json configs[2], the "collision-constrained"
workload the metric's target is stated on).  --config cfg1 drops the collision term (configs[1]); --config cfg3 is
configs[3] at its stated length (50 waypoints, CartVel + LVS continuous collision + via points; default 512 per GPU =
4096 / 8); --config cfg4 is configs[4] (14-DOF dual arm, 40 waypoints, upright constraints; default 256).

`value`  : inputs already resident in HBM (tb200_solve_batch_resident), device time = CUDA events on the solver's
           stream summed over the K steps, max over ranks.
`e2e`    : the same metric through the public API with HOST (pinned) buffers: H2D of the per-trajectory inputs and D2H
           of the results inside the timed region; the K steps are bracketed by ONE barrier + synchronize on each side
           (no per-step barrier), max over ranks.
Every step uses a different synthetic batch (seed = f(step, rank)), so nothing is cached between timed iterations; the
working set of one step (~0.6 GB of convexification rows + QP workspace at B=1024 with collision) is larger than L2.
--scaling strong splits ONE global batch (--batch) over the ranks instead of giving every rank its own.
--dump-outputs DIR writes the results of the last timed step of the `value` leg (what tb200_fetch_results hands the
caller) as DIR/<name>.npy in float64, so that two builds run with the same arguments can be compared output for output.
The benchmark writes nothing into the source tree.
"""
import argparse
import atexit
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from trajopt_b200 import problems  # noqa: E402

METRIC = "converged trajectories/sec (7-DOF x 30 wp, batch 1024)"
DEFAULT_BATCH = {"cfg1": 1024, "cfg2": 1024, "cfg3": 512, "cfg4": 256}


def batch_seed(it, rank, world):
    """Seed of the batch of step `it` on `rank`: both arms (and the parity spot check) build their batches from it."""
    return problems.SEED + 1 + 7919 * (it * world + rank)


def make_batch(config, batch, seed):
    if config == "cfg1":
        return problems.config1(B=batch, T=30, seed=seed)
    if config == "cfg2":
        return problems.config2(B=batch, T=30, seed=seed)
    if config == "cfg3":
        return problems.config3(B=batch, T=50, seed=seed)
    if config == "cfg4":
        return problems.config4(B=batch, T=40, seed=seed)
    raise SystemExit(f"unknown config {config}")


def workload_name(config, batch):
    if config == "cfg3":
        return (f"batch {batch} x 7-DOF x 50 waypoints, JointVel/JointAcc + CartPose via/terminal constraints + CartVel + "
                "LVS continuous collision (8 sphere obstacles, longest_valid_segment_length 0.05) = configs[3]")
    if config == "cfg4":
        return (f"batch {batch} x 14-DOF dual arm x 40 waypoints, JointVel/JointAcc + upright CartPose constraint per gripper "
                "and waypoint + terminal CartPose + discrete collision (14 x 8 spheres) = configs[4]")
    extra = " + discrete collision (8 sphere obstacles), safety_margin 0.02" if config == "cfg2" else ""
    return f"batch {batch} x 7-DOF x 30 waypoints, JointVel/JointAcc + CartPose terminal constraint{extra}"


def config_dict(args, world):
    """The `config` object of the JSON line: identical in both arms."""
    per_rank = args.batch // world if args.scaling == "strong" else args.batch
    return {"workload": workload_name(args.config, per_rank), "global_batch": per_rank * world,
            "parallelism": f"batch sharded over {world} GPU(s), no data-path collective",
            "timing": "fresh synthetic batch every step (seed = f(step, rank)); per-step working set > L2",
            "seeds": f"numpy default_rng({problems.SEED} + 1 + 7919 * (step * world + rank))"}


# ---------------------------------------------------------------------------------------------------------- host info
def host_info():
    """What the CPU arm runs on: logical CPUs, physical cores, the CPUs this process may use, the cgroup CPU quota,
    the CPU model and the load when the measurement starts (two boxes of one pool have differed 3.5x in round 1)."""
    info = {"logical_cpus": os.cpu_count()}
    try:
        info["affinity"] = len(os.sched_getaffinity(0))
    except AttributeError:
        info["affinity"] = info["logical_cpus"]
    try:
        import psutil
        info["physical_cores"] = psutil.cpu_count(logical=False)
    except ImportError:
        info["physical_cores"] = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            info["cgroup_cpu_max"] = open(path).read().strip()
            break
        except OSError:
            continue
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                info["cpu_model"] = line.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    try:
        info["loadavg"] = os.getloadavg()[0]
    except OSError:
        pass
    return info


def host_threads(info=None):
    """Host threads of the CPU legs: one per physical core this process may run on, capped by the cgroup CPU quota
    (torchrun exports OMP_NUM_THREADS=1, which must not shrink the CPU baseline).  Measured on the GPU box in round 1
    (2 x 64 hardware threads), full batch of 1024: 64 threads 6.3 s, 128 threads 8.5 s - the oracle is bound by its
    allocator and caches, SMT siblings only hurt."""
    if os.environ.get("TB200_CPU_THREADS"):
        return int(os.environ["TB200_CPU_THREADS"])
    info = info or host_info()
    n = info.get("affinity") or info.get("logical_cpus") or 1
    if info.get("physical_cores"):
        n = min(n, info["physical_cores"])
    quota = info.get("cgroup_cpu_max", "")
    parts = quota.split()
    if len(parts) == 2 and parts[0].isdigit() and parts[1].isdigit() and int(parts[1]) > 0:
        n = min(n, max(1, int(parts[0]) // int(parts[1])))
    return max(1, n)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                          str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            atexit.register(self.proc.kill)  # the sampler must not outlive a run that raises before stop()
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(s[0]) for s in self.samples if s and s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(s) > 2 + i and s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons}


# ------------------------------------------------------------------------------------------------------------ CPU arm
def oracle_module():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib  # the CPU legs: the oracle is the timed CPU path here, never part of the product
    oracle_lib.lib()  # loads the library build() made; no make run, so a read-only tree works
    return oracle_lib


def cpu_time(oracle_lib, desc, threads, b1=None, repeats=1):
    """Best of `repeats` oracle solves of desc[0:b1]: (seconds, converged)."""
    best, conv = None, 0
    for _ in range(repeats):
        t0 = time.perf_counter()
        r = oracle_lib.solve_batch(desc, 0, b1, n_threads=threads)
        dt = time.perf_counter() - t0
        n = desc.B if b1 is None else b1
        if best is None or dt < best:
            best, conv = dt, int((r["status"][:n] == 0).sum())
    return best, conv


def cpu_sweep(oracle_lib, desc, threads):
    """Thread scaling of the CPU path on a small sample (explains the quoted number: does the box deliver its cores?)
    and the single-thread latency per trajectory."""
    out = {}
    t1, _ = cpu_time(oracle_lib, desc, 1, b1=min(16, desc.B))
    out["single_thread_s_per_trajectory"] = t1 / min(16, desc.B)
    n = min(128, desc.B)
    for th in sorted({8, 32, threads}):
        if th > threads:
            continue
        dt, _ = cpu_time(oracle_lib, desc, th, b1=n)
        out[f"trajectories_per_s_{th}_threads"] = n / dt
    out["sample"] = f"{n} trajectories (16 for the single thread)"
    return out


def run_reference(args, rank, world):
    """CPU arm: the reference's own CPU path restated (oracle/; the reference cannot be compiled here: no Eigen / OSQP /
    tesseract, DESIGN.md), OpenMP over trajectories on the host cores, on rank 0's batches of the CUDA arm (same seeds).
    Mode: reference-faithful, i.e. the QP is set up from scratch (scaling + factorisation) on every Model::optimize()
    call, as OSQPModel does with update_workspace == false (osqp_interface.cpp:283-370)."""
    if rank != 0:
        return
    oracle_lib = oracle_module()
    info = host_info()
    threads = host_threads(info)
    per_rank = args.batch // world if args.scaling == "strong" else args.batch
    sample = min(args.cpu_sample, per_rank) if args.cpu_sample else per_rank
    times, conv = [], []
    for it in range(args.warmup + args.steps):
        desc = make_batch(args.config, per_rank, batch_seed(it, 0, world))
        dt, c = cpu_time(oracle_lib, desc, threads, b1=sample)
        if it >= args.warmup:
            times.append(dt)
            conv.append(c)
    value = sum(conv) / sum(times)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "trajectories/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * float(np.mean(times)), "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(args, world),
            "cpu_baseline": {"value": value, "unit": "trajectories/s", "cores": threads, "kind": "port",
                             "mode": "reference-faithful (QP re-setup on every optimize(), osqp_interface.cpp:283-370)",
                             "sample": f"the first {sample} trajectories of every step's batch, OpenMP over trajectories; "
                                       f"best step {min(times):.2f} s, worst {max(times):.2f} s",
                             "best_step_value": max(c / t for c, t in zip(conv, times)), "host": info},
            "e2e": {"value": value, "unit": "trajectories/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------- CUDA arm
def measured_traffic(config):
    """dram__bytes_read.sum + dram__bytes_write.sum of one full-batch convexify launch from this round's
    `ncu --set full` capture (profiles/r02_convexify_ncu.json, written by scripts/ncu_traffic.py); None without one."""
    path = os.path.join(ROOT, "profiles", "r02_convexify_ncu.json")
    try:
        d = json.load(open(path))
        return d.get(config, {}).get("dram_bytes")
    except (OSError, ValueError):
        return None


DUMP_BUDGET = 64 << 20


def dump_outputs(out_dir, res, budget=DUMP_BUDGET):
    """Writes the per-trajectory result arrays of one solve as out_dir/<name>.npy (float64).  Above `budget` bytes a fixed
    sample of trajectories (numpy default_rng(0), in batch order) is written instead, with their batch indices in
    trajectory_index.npy."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in res.items() if isinstance(v, np.ndarray)}
    B = len(arrays["status"])
    per_traj = sum(a.nbytes for a in arrays.values()) / B + 8
    n = min(B, int((budget - 128 * (len(arrays) + 1)) // per_traj))  # 128: one .npy header per file
    if n < B:
        idx = np.sort(np.random.default_rng(0).choice(B, n, replace=False))
        arrays = {k: a[idx] for k, a in arrays.items()}
        arrays["trajectory_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--config", default="cfg2", choices=["cfg1", "cfg2", "cfg3", "cfg4"])
    ap.add_argument("--batch", type=int, default=0, help="trajectories per GPU (weak scaling) / in total (strong scaling); "
                                                         "default: the config's stated size")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--cpu-sample", type=int, default=0,
                    help="trajectories per CPU step (default 0: one whole batch, so that the CPU path is bound by its "
                         "longest trajectory exactly as the GPU path is)")
    ap.add_argument("--cpu-repeats", type=int, default=3, help="cpu_baseline: best of this many runs")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step as DIR/<name>.npy "
                                                          f"(float64, at most {DUMP_BUDGET >> 20} MB in all)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs writes the results of the CUDA path (--impl cuda)")
    if args.batch <= 0:
        args.batch = DEFAULT_BATCH[args.config]

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl cuda needs a CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from trajopt_b200 import api, capi

    # each rank owns its own independent trajectories (shards never interact: no data-path collective)
    per_rank = args.batch // world if args.scaling == "strong" else args.batch
    total = args.warmup + args.steps
    if args.scaling == "strong":  # ONE global batch per step, rank r takes its contiguous shard
        from trajopt_b200 import sharding
        batches = []
        for it in range(total):
            g = make_batch(args.config, per_rank * world, batch_seed(it, 0, 1))
            lo, hi = rank * per_rank, (rank + 1) * per_rank
            batches.append(capi.ProblemDesc(g.robot_spec, g.T, g.terms, g.init_traj[lo:hi], fixed_timesteps=list(g._fixed_t),
                                            cart_targets=g.cart_targets[lo:hi], obstacles=None if g.obstacles is None else g.obstacles[lo:hi]))
    else:
        batches = [make_batch(args.config, per_rank, batch_seed(it, rank, world)) for it in range(total)]
    prob = api.Problem(batches[0], device=local_rank)
    pinned = [dict(init=torch.from_numpy(b.init_traj).pin_memory(), tgt=torch.from_numpy(b.cart_targets).pin_memory(),
                   obs=None if b.obstacles is None else torch.from_numpy(b.obstacles).pin_memory()) for b in batches]

    def fence():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ptr = lambda t: None if t is None else capi.C.cast(t.data_ptr(), capi.C.POINTER(capi.C.c_double))

    def step_resident(it):
        pb = pinned[it]
        prob._check(prob.lib.tb200_problem_set_inputs(prob.handle, ptr(pb["init"]), ptr(pb["tgt"]), ptr(pb["obs"])))
        torch.cuda.synchronize()
        prob.solve_resident()
        tm = prob.timing()
        return tm, prob.fetch()

    def step_e2e(it):
        pb = pinned[it]
        prob._check(prob.lib.tb200_problem_set_inputs(prob.handle, ptr(pb["init"]), ptr(pb["tgt"]), ptr(pb["obs"])))
        return prob.solve()

    sampler = ClockSampler(local_rank)
    # ---- resident leg (value): device time per step from CUDA events on the solver's stream -------------------------
    for it in range(args.warmup):
        step_resident(it)
    fence()
    if rank == 0:
        sampler.start()
    dev_ms, conv, tms, ktm = [], [], [], []
    for it in range(args.warmup, total):
        tm, res = step_resident(it)
        dev_ms.append(tm["total_ms"])
        conv.append(int((res["status"] == 0).sum()))
        tms.append(tm)
        # the convexify kernel alone, every trajectory active, at this step's solution (new data every launch; one
        # launch writes ~135 MB > L2): the launch the roofline below is quoted on
        ktm.append(prob.convexify_timed(res["x"]))
    fence()
    resident_last = res
    # ---- end-to-end leg: K steps through the public API with host buffers, one fence on each side -------------------
    t0 = time.perf_counter()
    e2e_conv, h2d, d2h, last = 0, 0, 0, None
    for it in range(args.warmup, total):
        res = step_e2e(it)
        e2e_conv += int((res["status"] == 0).sum())
        h2d, d2h = res["timing"]["h2d_bytes"], res["timing"]["d2h_bytes"]
        last = res
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    clocks = sampler.stop() if rank == 0 else None
    fence()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs if world == 1 else os.path.join(args.dump_outputs, f"rank{rank}"), resident_last,
                     DUMP_BUDGET // world)

    def reduce(v, op):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=op)  # report only: the data path has no collective
        return float(t.item())

    MAX, SUM = (dist.ReduceOp.MAX, dist.ReduceOp.SUM) if world > 1 else (None, None)
    dev_total_s = reduce(sum(dev_ms) / 1e3, MAX)     # device time (CUDA events on the solver stream), max over ranks
    conv_total = reduce(float(sum(conv)), SUM)
    e2e_total_s = reduce(e2e_s, MAX)
    e2e_conv_total = reduce(float(e2e_conv), SUM)
    # the batches of every rank, step by step: a batch is as slow as its longest trajectory (tens of thousands of
    # dependent ADMM iterations), so its time varies with the draw — the spread is part of the measurement
    step_ms_min, step_ms_max = reduce(-min(dev_ms), MAX), reduce(max(dev_ms), MAX)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    value = conv_total / dev_total_s
    # ---- roofline of the convexify kernel (HBM bound; algorithmic bytes per launch: DESIGN.md section 4) -------------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (burst)"
    conv_ms = sum(t["convexify_ms"] for t in tms)
    conv_launches = sum(t["convexify_launches"] for t in tms)
    k_ms = sum(t["convexify_ms"] for t in ktm)
    k_bytes = sum(t["convexify_bytes"] for t in ktm)
    achieved = k_bytes / (k_ms * 1e-3) / 1e9 if k_ms > 0 else 0.0
    roofline = {"bound": "hbm", "kernel": "eval_convexify_decide_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": measured_traffic(args.config), "peak_source": peak_src,
                "scope": "one full-batch launch per timed step (all trajectories active), CUDA events on the launching stream",
                "avg_launch_us": 1e3 * k_ms / max(len(ktm), 1), "algorithmic_bytes_per_launch": k_bytes / max(len(ktm), 1),
                "in_step": {"share_of_step": conv_ms / (sum(dev_ms)), "evaluations": conv_launches,
                            "note": "inside a solve the same code runs as a step of the persistent solve_kernel, one "
                                    "trajectory per CTA at a time (share = SM time in evaluation steps, %globaltimer)"}}
    qp_ms = sum(t["qp_ms"] for t in tms)
    line = {"metric": METRIC, "value": value, "unit": "trajectories/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dev_total_s / args.steps, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(args, world),
            "converged_fraction": conv_total / (per_rank * world * args.steps),
            "e2e": {"value": e2e_conv_total / e2e_total_s, "unit": "trajectories/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": 1e3 * e2e_total_s / args.steps},
            # per solve: reset_state_kernel, eval_convexify_decide_kernel (initial evaluation), solve_kernel (persistent);
            # plus the stand-alone convexify launch the roofline is quoted on (resident leg only)
            "ms_per_step_rank0": [round(x, 1) for x in dev_ms],
            "ms_per_step_spread": {"min_over_ranks_and_steps": round(-step_ms_min, 1), "max_over_ranks_and_steps": round(step_ms_max, 1),
                                   "note": "a batch is bound by its longest trajectory: the time of a fresh batch varies with the draw"},
            "gpu_launches": 4 * len(tms) + 3 * args.steps,
            "roofline": roofline,
            "qp_steps": {"share_of_step": qp_ms / sum(dev_ms), "qp_solves": int(sum(t["qp_launches"] for t in tms)),
                         "note": "QP steps of solve_kernel (ADMM): shared-memory/latency bound, see profiles/ for achieved occupancy"},
            "clocks": clocks}
    oracle_lib = None
    if not args.no_parity:
        # parity spot check outside the timed region: 32 trajectories of the LAST timed batch against the CPU oracle
        oracle_lib = oracle_module()
        n = min(32, per_rank)
        ref = oracle_lib.solve_batch(batches[total - 1], 0, n, n_threads=host_threads())
        line["parity"] = {"n": n, "status_match": bool((last["status"][:n] == ref["status"][:n]).all()),
                          "qp_count_match": bool((last["n_qp_solves"][:n] == ref["n_qp_solves"][:n]).all()),
                          "max_dcost": float(np.abs(last["total_cost"][:n] - ref["total_cost"][:n]).max()),
                          "max_dx": float(np.abs(last["x"][:n] - ref["x"][:n]).max()),
                          "against": "CPU oracle on the same inputs (first trajectories of the last timed batch)"}
    if not args.no_cpu_baseline:
        oracle_lib = oracle_lib or oracle_module()
        info = host_info()
        threads = host_threads(info)
        desc = batches[total - 1]  # the last timed batch: the CPU path gets byte-identical inputs
        sample = min(args.cpu_sample, per_rank) if args.cpu_sample else per_rank
        dt, c = cpu_time(oracle_lib, desc, threads, b1=sample, repeats=max(1, args.cpu_repeats))
        line["cpu_baseline"] = {"value": c / dt, "unit": "trajectories/s", "cores": threads, "kind": "port",
                                "mode": "reference-faithful (QP re-setup on every optimize(), osqp_interface.cpp:283-370)",
                                "sample": f"the first {sample} trajectories of the last timed batch, best of "
                                          f"{max(1, args.cpu_repeats)} runs: {dt:.2f} s", "host": info,
                                "sweep": cpu_sweep(oracle_lib, desc, threads)}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
