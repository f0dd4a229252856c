#!/usr/bin/env python
"""bench.py -- batched MPC solve throughput of the B200 engine (and the CPU reference arm).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--problems B] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR: after the timed steps, rank 0 writes what its last timed step returned -- plan [H][2][B],
losses [S][B] and best [B] (the winning start, as float32) -- to DIR/<name>.npy.  The inputs are seeded, so the same
arguments give the same problems on every run and two builds can be compared output for output.  Above 64 MB in all
a fixed, seeded sample of problems is written, with their indices in DIR/problem_index.npy.

One step = one pass of the hot path over one batch: ONE ocd_solve_batch launch that runs
NaivePlanner.generate_plan (3 starts x 100 SGD iterations + final losses + argmin) for B
independent problems of the finite_horizon shape (H=5, 2 cars, 3 lanes).  Rank r solves its own
B problems (weak scaling, no data-path collective: the problems are independent); the value is
all ranks' solves divided by the slowest rank's device time.

Extra keys on the JSON line: roofline (FP32-pipe bound; the peak is measured in this job with a
dependent-free FMA kernel, since MEASURED_PEAKS.json has no FP32 figure), hbm (algorithmic bytes
vs the measured copy bandwidth, to show the path is nowhere near memory-bound), e2e (same metric
through the host-buffer C ABI, copies inside), cpu_baseline (the CPU oracle on this box's cores),
cmaes (candidate-evals/s of one CMA-ES generation of BASELINE configs[1..3]: finite_horizon n_inits 5, local_opt
n_inits 10, replanning T=20 x 2 samples -- one episode launch each), cmaes_dropin (the first of them through the
MPC_ORD drop-in, host wall clock), cmaes_multi_dropin (64 lock-step runs through optimize_cmaes_lockstep, host wall
clock), cmaes_multi (64 independent CMA-ES runs per GPU in
lock step: the axis on which candidate-evals/s scales with GPUs), horizons (solves/s at H = 15 and H = 50, the other
horizons BASELINE's metric names), sweep (corner points of BASELINE configs[4]), e2e_first_control (the
receding-horizon caller's host call: only plan[0] comes back), cpu_baseline_serial (the reference's own driving style:
one problem at a time, one autograd call per SGD step, one thread).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True           # the bench writes nothing into the tree it runs from (it may be read-only)

SHAPE = dict(H=5, C=2, L=3, S=3, n_iter=100)
METRIC, UNIT = "mpc_solves_per_sec", "solves/s"
DUMP_LIMIT = 64 * 10**6                  # bytes --dump-outputs may write, .npy headers included


def dump_outputs(out_dir: str, out: dict, B: int) -> None:
    """Writes one step's device outputs (problem axis last) as float32 .npy files under out_dir; above DUMP_LIMIT
    a fixed, seeded sample of the problems, whose indices go to problem_index.npy (float64, exact)."""
    host = {k: v.cpu().numpy() for k, v in out.items()}
    host["best"] = host["best"].astype(np.float32)            # start indices 0..5: exact in float32
    per_problem = sum(a.nbytes for a in host.values()) // B
    if per_problem * B > DUMP_LIMIT - 4096:
        n = (DUMP_LIMIT - 4096) // (per_problem + 8)          # + the float64 index of each kept problem
        sel = np.sort(np.random.default_rng(0).choice(B, n, replace=False))
        host = {k: np.ascontiguousarray(a[..., sel]) for k, a in host.items()}
        host["problem_index"] = sel.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in host.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), a)


def _config(B, n_gpus, per_step=None):
    """per_step: problems one step actually solves when that is a bounded sample of the workload (the CPU arm)."""
    cfg = {"workload": "synthetic sweep (BASELINE configs[4]) at the finite_horizon shape: independent MPC problems, "
                       "H=5, 2 cars, 3 lanes, 3 starts x 100 SGD iterations",
           "problems_per_gpu": B, "n_gpus": n_gpus, "horizon": 5, "cars": 2, "lanes": 3, "starts": 3,
           "n_iter": 100, "lr": 0.1, "inits_per_candidate": 5, "parallelism": f"problem-sharded x{n_gpus}",
           "l2_policy": "4 rotating input/output sets (>= 350 MB in total, L2 is 126 MB)"}
    if per_step is not None:
        cfg["problems_per_step"] = per_step
        cfg["sample_note"] = (f"the CPU arm solves a bounded sample of {per_step} problems of this workload per step on the "
                              f"host, not {B} per GPU; solves/s is a rate, so the two arms compare directly")
        cfg["l2_policy"] = "n/a (host)"
    return cfg


# ---------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU during the timed region (NVML)."""

    def __init__(self, index: int, period: float = 0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40,
                 "sw_thermal_slowdown": 0x20, "hw_power_brake_slowdown": 0x80}
        while not self._halt.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        med = int(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def _visible_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


# ---------------------------------------------------------------------------------------------
def host_threads() -> int:
    """Host cores this process may use.  (torchrun exports OMP_NUM_THREADS=1; the oracle's OpenMP loop
    takes its thread count as an argument, so that default does not throttle the CPU arm.)"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def cpu_arm(problems: int, threads: int | None = None, seed: int = 1234):
    """Times the CPU oracle (oracle/: C restatement of the reference's planner, OpenMP over
    problems) on `problems` synthetic problems of the bench shape.  -> (solves/s, seconds, threads)"""
    import oracle as O
    from l4dc_mpc_ocd_b200 import synthetic       # plain numpy; the package loads libocd_b200.so only when the engine is used
    threads = threads or host_threads()
    batch = synthetic.make_batch(problems, seed=seed)
    w = batch["weights"][batch["weight_idx"]]
    p = O.OracleParams()
    t0 = time.perf_counter()
    O.generate_plan_batch(p, batch["world"], w, nthreads=threads)
    dt = time.perf_counter() - t0
    return problems / dt, dt, threads


def reference_main(args, rank: int, world_size: int):
    """--impl reference: the reference planner's CPU implementation on this box's host cores.
    TensorFlow (the reference's substrate) is not installable here, so the timed code is the
    oracle port of NaivePlanner.generate_plan, all host threads (cpu_baseline.kind = "port")."""
    if rank != 0:
        return
    threads = host_threads()
    rate, _, _ = cpu_arm(max(256, 32 * threads), threads)          # calibrate
    per_step = int(max(256, min(rate * 1.5, 2_000_000)))           # about 1.5 s of CPU work per step
    for _ in range(args.warmup):
        cpu_arm(max(256, per_step // 8), threads)
    t_tot = 0.0
    for i in range(args.steps):
        _, dt, _ = cpu_arm(per_step, threads, seed=1234 + i)
        t_tot += dt
    value = per_step * args.steps / t_tot
    cfg = _config(args.problems, args.gpus, per_step=per_step)
    sample = f"{per_step} synthetic problems of the bench shape per step x {args.steps} steps"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }), flush=True)


# ---------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--problems", type=int, default=1 << 20, help="MPC problems per GPU per step")
    ap.add_argument("--no-extras", action="store_true", help="skip e2e / cpu_baseline / cmaes legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world_size = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        reference_main(args, rank, world_size)
        return

    import torch
    import torch.distributed as dist
    import l4dc_mpc_ocd_b200 as ocd
    from l4dc_mpc_ocd_b200 import synthetic

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    from l4dc_mpc_ocd_b200 import parallel
    # one process per GPU on one host: each rank takes its own slice of the host's cores (copy threads, pinned buffers)
    cpus_owned = parallel.bind_rank_cpus(local_rank, int(os.environ.get("LOCAL_WORLD_SIZE", world_size)))
    distributed = world_size > 1
    if distributed:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    eng = ocd.Engine(local_rank)
    dev = eng.device
    B, K, W = args.problems, args.steps, args.warmup
    p = ocd.PlannerParams()                  # finite_horizon shape, fast-math kernels

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x: float) -> float:
        if not distributed:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # inputs resident in HBM, SoA; 4 rotating sets so that no step finds its data in L2
    NSETS = 4
    sets = []
    for i in range(NSETS):
        b = synthetic.make_batch(B, seed=1234 + 17 * rank + i)
        world = torch.as_tensor(b["world"], device=dev).permute(1, 2, 0).contiguous()
        weights = torch.as_tensor(b["weights"], device=dev).t().contiguous()
        idx = torch.as_tensor(b["weight_idx"], device=dev)
        out = dict(plan=torch.empty((p.H, 2, B), dtype=torch.float32, device=dev),
                   losses=torch.empty((p.S, B), dtype=torch.float32, device=dev),
                   best=torch.empty((B,), dtype=torch.int32, device=dev))
        sets.append((world, weights, idx, out, b))
    Bw = sets[0][1].shape[1]

    def step(i):
        world, weights, idx, out, _ = sets[i % NSETS]
        eng.solve_soa(p, world, weights, Bw, idx, out=out)

    fp32_peak = eng.fp32_peak(8192)          # roofline denominator, measured before the run
    for i in range(W):
        step(i)
    barrier()
    sampler = ClockSampler(_visible_index(local_rank))
    sampler.start()
    launches0 = eng.kernel_launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        step(W + i)
    e1.record()
    barrier()
    ms_total = max_over_ranks(float(e0.elapsed_time(e1)))
    clocks = sampler.stop()
    launches = eng.kernel_launches - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, sets[(W + K - 1) % NSETS][3], B)
    value = B * K * world_size / (ms_total * 1e-3)
    ms_per_step = ms_total / K

    # roofline of the dominant (only) kernel: k_solve
    flops = synthetic.flops_per_solve(SHAPE["H"], SHAPE["C"], SHAPE["L"], SHAPE["S"], SHAPE["n_iter"])
    hbm_bytes = synthetic.hbm_bytes_per_solve(SHAPE["H"], SHAPE["C"], SHAPE["L"], SHAPE["S"])
    own_ms = float(e0.elapsed_time(e1)) / K
    achieved_tf = flops * B / (own_ms * 1e-3) / 1e12
    peaks = {}
    try:
        peaks = json.load(open(ROOT / "MEASURED_PEAKS.json"))
    except Exception:
        pass
    traffic = None
    try:
        traffic = json.load(open(ROOT / "profiles" / "traffic.json")).get("k_solve_bytes_per_launch")
    except Exception:
        pass
    nominal_tf = 148 * 128 * 2 * (clocks.get("sm_max_mhz") or 1965) * 1e6 / 1e12
    roofline = {"bound": "fp32", "achieved": achieved_tf, "peak": fp32_peak / 1e12, "unit": "TFLOP/s",
                "frac": achieved_tf / (fp32_peak / 1e12), "traffic": traffic,
                "bound_note": "BASELINE's north_star names the FP32 pipe as this path's roofline: no stage is a dense "
                              "contraction (no tensor roofline) and HBM carries 0.3 % of its measured bandwidth (see hbm)",
                "peak_source": "dependent-free FFMA kernel (512 FMAs per loop trip) measured in this job; "
                               "MEASURED_PEAKS.json has no FP32 figure; nominal = 148 SMs x 128 lanes x 2 x sm_max_mhz",
                "nominal_peak": nominal_tf, "frac_of_nominal": achieved_tf / nominal_tf,
                "flops_per_solve": flops, "kernel": f"k_solve<5,1,3,fast,{ocd.kernel_form(p, B)}>", "kernel_ms": own_ms,
                "traffic_source": "profiles/traffic.json: dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set "
                                  "full capture of this kernel at this batch size (not re-measured in this job)"}
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    hbm = {"achieved": hbm_bytes * B / (own_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
           "peak_source": "MEASURED_PEAKS.json (measured)" if "hbm_gbs" in peaks else "fallback",
           "bytes_per_solve": hbm_bytes}
    hbm["frac"] = hbm["achieved"] / hbm_peak

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world_size, "steps": K, "warmup": W,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": _config(B, world_size), "clocks": clocks,
            "gpu_launches": launches, "roofline": roofline, "hbm": hbm}

    # ---- e2e: the same solves through the host-buffer C ABI (ocd_solve_batch_host) ----------------
    # inputs start in pinned host memory, results end in pinned host memory; every step pays the
    # host->device copy of its inputs and the device->host copy of plans, losses and winners.
    if not args.no_extras:
        ctx = ocd.HostContext(local_rank)
        hb = sets[0][4]

        def pinned(a):
            buf = ocd.HostContext.pinned_empty(a.shape, a.dtype)
            buf[...] = a
            return buf

        h_world = pinned(np.ascontiguousarray(hb["world"].transpose(1, 2, 0)))
        h_w = pinned(np.ascontiguousarray(hb["weights"].T))
        h_idx = pinned(hb["weight_idx"])
        h_out = dict(plan=ocd.HostContext.pinned_empty((p.H, 2, B)), losses=ocd.HostContext.pinned_empty((p.S, B)),
                     best=ocd.HostContext.pinned_empty((B,), np.int32))
        ke = max(3, min(K, 10))
        for _ in range(2):
            ctx.solve_soa(p, h_world, h_w, weight_idx=h_idx, out=h_out)
        barrier()
        t0 = time.perf_counter()
        for _ in range(ke):
            r = ctx.solve_soa(p, h_world, h_w, weight_idx=h_idx, out=h_out)
        t_e2e = max_over_ranks(time.perf_counter() - t0)
        # the same call on ordinary pageable numpy arrays (staged through the context's pinned area)
        # (outputs too: ordinary numpy arrays reused across steps, as a steady-state caller would)
        pg_world, pg_w, pg_idx = np.array(h_world), np.array(h_w), np.array(h_idx)
        pg_out = {k: np.zeros_like(v) for k, v in h_out.items()}
        ctx.solve_soa(p, pg_world, pg_w, weight_idx=pg_idx, out=pg_out)
        barrier()
        t0 = time.perf_counter()
        for _ in range(3):
            ctx.solve_soa(p, pg_world, pg_w, weight_idx=pg_idx, out=pg_out)
        t_pageable = max_over_ranks(time.perf_counter() - t0) / 3
        # ... and the same ordinary arrays page-locked in place once (ocd_host_register): what a steady-state caller
        # that reuses its arrays does -- the copy engines then work on them directly, no staging memcpy
        regs, done_regs, t_registered = [pg_world, pg_w, pg_idx] + list(pg_out.values()), [], None
        try:
            for a in regs:
                ocd.HostContext.register(a)
                done_regs.append(a)
            reg_ok = 1.0
        except Exception:                     # a host that refuses to page-lock that much: report the leg as absent
            reg_ok = 0.0
        if distributed:                       # every rank takes the same branch
            t = torch.tensor([reg_ok], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            reg_ok = float(t.item())
        if reg_ok:
            ctx.solve_soa(p, pg_world, pg_w, weight_idx=pg_idx, out=pg_out)
            barrier()
            t0 = time.perf_counter()
            for _ in range(ke):
                ctx.solve_soa(p, pg_world, pg_w, weight_idx=pg_idx, out=pg_out)
            t_registered = max_over_ranks(time.perf_counter() - t0) / ke
        for a in done_regs:
            ocd.HostContext.unregister(a)
        line["e2e"] = {"value": B * ke * world_size / t_e2e, "unit": UNIT,
                       "h2d_bytes_per_step": int(h_world.nbytes + h_w.nbytes + h_idx.nbytes),
                       "d2h_bytes_per_step": int(r["plan"].nbytes + r["losses"].nbytes + r["best"].nbytes),
                       "steps": ke, "ms_per_step": 1e3 * t_e2e / ke,
                       "api": "ocd_solve_batch_host: pinned host arrays in, pinned host arrays out, "
                              "ramped column chunks over an H2D stream, two compute lanes and a D2H stream, so copies overlap the solve",
                       "pageable_host_arrays_value": B * world_size / t_pageable,
                       "registered_host_arrays_value": None if t_registered is None else B * world_size / t_registered}
        # the receding-horizon caller's call (ocd_solve_first_host): same inputs, only plan[0] + losses + winner come back
        f_out = dict(first=ocd.HostContext.pinned_empty((2, B)), losses=h_out["losses"], best=h_out["best"])
        for _ in range(2):
            ctx.solve_first_soa(p, h_world, h_w, weight_idx=h_idx, out=f_out)
        barrier()
        t0 = time.perf_counter()
        for _ in range(ke):
            ctx.solve_first_soa(p, h_world, h_w, weight_idx=h_idx, out=f_out)
        t_first = max_over_ranks(time.perf_counter() - t0)
        line["e2e_first_control"] = {
            "value": B * ke * world_size / t_first, "unit": UNIT, "ms_per_step": 1e3 * t_first / ke,
            "h2d_bytes_per_step": line["e2e"]["h2d_bytes_per_step"],
            "d2h_bytes_per_step": int(f_out["first"].nbytes + f_out["losses"].nbytes + f_out["best"].nbytes),
            "api": "ocd_solve_first_host: what PlannerCar._get_next_control needs -- plan[0], losses, winner"}
        line["e2e"]["host_cpus_per_rank"] = cpus_owned
        line["gpu_launches"] = launches
        ctx.close()

        # ---- candidate-evals/s: one CMA-ES generation of finite_horizon cmaes --n_inits 5 -------------
        dd = dist if distributed else None
        line["cmaes"] = cmaes_leg(eng, ocd, dd, rank, world_size, max_over_ranks, barrier, "finite_horizon", 5)
        line["cmaes_configs"] = [line["cmaes"],
                                 cmaes_leg(eng, ocd, dd, rank, world_size, max_over_ranks, barrier, "local_opt", 10),
                                 cmaes_leg(eng, ocd, dd, rank, world_size, max_over_ranks, barrier, "replanning", 5)]
        if world_size == 1:
            line["cmaes_dropin"] = cmaes_dropin_leg()
        line["cmaes_multi_dropin"] = cmaes_multi_dropin_leg(world_size, max_over_ranks, barrier)
        # independent CMA-ES runs in lock step: 64 runs per GPU (weak), and a fixed 512 runs over all GPUs (strong)
        line["cmaes_multi"] = cmaes_leg(eng, ocd, dd, rank, world_size, max_over_ranks, barrier, "finite_horizon", 5,
                                        runs=64 * world_size)
        line["cmaes_multi_strong"] = cmaes_leg(eng, ocd, dd, rank, world_size, max_over_ranks, barrier, "finite_horizon",
                                               5, runs=512)

        # ---- the other horizons of the metric (H = 5..50): two points of BASELINE configs[4] -------------------
        line["horizons"] = horizons_leg(eng, ocd, synthetic, rank, world_size, max_over_ranks, barrier, fp32_peak,
                                        nominal_tf * 1e12)
        # ---- BASELINE configs[4]: corner points of the sweep (all of it: scripts/sweep.py -> profiles/) ----------
        line["sweep"] = sweep_leg(eng, ocd, synthetic, rank, world_size, max_over_ranks, barrier, nominal_tf * 1e12)

    # ---- CPU baseline beside it (rank 0, N=1 only) -------------------------------------------------
    if not args.no_extras and world_size == 1:
        threads = host_threads()
        rate, _, _ = cpu_arm(max(256, 32 * threads), threads)
        n = int(max(512, min(rate * 12.0, 4_000_000)))         # about 12 s of CPU work
        v, dt, _ = cpu_arm(n, threads)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                                "sample": f"{n} problems of the bench shape, oracle C port with OpenMP, {dt:.1f} s"}
        # the reference's own driving style (BASELINE.md section 3, cpu_ref_serial): one problem at a time, a Python
        # loop with one autograd call per SGD step, one thread -- torch-CPU standing in for TensorFlow
        from oracle import torch_serial
        vs, dts = torch_serial.time_serial_solves(2)
        line["cpu_baseline_serial"] = {"value": vs, "unit": UNIT, "cores": 1, "kind": "port",
                                       "sample": f"2 problems of the bench shape, float32 torch-CPU autograd restatement "
                                                 f"driven like the reference (one tape per SGD step), {dts:.1f} s"}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if distributed:
        dist.destroy_process_group()


SWEEP_LR = {5: 0.1, 15: 0.02, 50: 0.0003}     # the reference's lr = 0.1 is only stable at its own H = 5 / 6


def _timed_solve(eng, ocd, synthetic, rank, world_size, max_over_ranks, barrier, H, C, B, reps):
    """One sweep point, device-resident: -> (ms per launch as the max over ranks, all losses finite)."""
    import torch
    p = ocd.PlannerParams(H=H, C=C, lr=SWEEP_LR.get(H, 0.1))
    b = synthetic.make_batch(B, C=C, seed=99 + rank)
    world = torch.as_tensor(b["world"], device=eng.device).permute(1, 2, 0).contiguous()
    w = torch.as_tensor(b["weights"], device=eng.device).t().contiguous()
    idx = torch.as_tensor(b["weight_idx"], device=eng.device)
    out = eng.solve_soa(p, world, w, w.shape[1], idx)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        eng.solve_soa(p, world, w, w.shape[1], idx, out=out)
    e1.record()
    barrier()
    ms = max_over_ranks(float(e0.elapsed_time(e1))) / reps
    finite = bool(torch.isfinite(out["losses"]).all().item())
    return p, ms, finite


def horizons_leg(eng, ocd, synthetic, rank, world_size, max_over_ranks, barrier, fp32_peak, nominal):
    """H = 15 and H = 50 (2 cars, the sweep's learning rates), device-resident, a few launches each: the
    medium-horizon (Q) and long-horizon (segmented) kernels.  Same accounting as the headline: all ranks'
    solves / slowest rank's time."""
    rows = []
    # 2^20 problems per GPU like the headline (BASELINE configs[4]'s largest batch): 32 768 blocks are hundreds of
    # waves, so the tail of the last wave does not colour the figure (at 65 536 problems H = 50 runs 3.46 waves of
    # four blocks per SM and loses 13 % to the tail alone; the small batches are in the `sweep` key)
    for H, B, reps in ((15, 1048576, 4), (50, 1048576, 2)):
        p, ms, finite = _timed_solve(eng, ocd, synthetic, rank, world_size, max_over_ranks, barrier, H, 2, B, reps)
        fl = synthetic.flops_per_solve(H, 2, 3)
        rows.append({"horizon": H, "problems_per_gpu": B, "lr": p.lr, "ms_per_launch": ms,
                     "solves_per_sec": B * world_size / (ms * 1e-3), "kernel_form": ocd.kernel_form(p, B),
                     "frac_of_measured_fp32": fl * B / (ms * 1e-3) / fp32_peak,
                     "frac_of_nominal_fp32": fl * B / (ms * 1e-3) / nominal, "all_losses_finite": finite})
    return rows


def sweep_leg(eng, ocd, synthetic, rank, world_size, max_over_ranks, barrier, nominal):
    """Corner points of BASELINE configs[4] (4K..1M problems x H 5/15/50 x 2..6 cars), per GPU, all ranks at once."""
    rows = []
    for H in (5, 15, 50):
        for C in (2, 6):
            for B in (4096, 1048576):
                reps = 2 if H * B >= 15 * 1048576 else 5
                p, ms, finite = _timed_solve(eng, ocd, synthetic, rank, world_size, max_over_ranks, barrier, H, C, B, reps)
                fl = synthetic.flops_per_solve(H, C, 3)
                rows.append({"H": H, "C": C, "B_per_gpu": B, "lr": p.lr, "ms": round(ms, 4),
                             "solves_per_sec": B * world_size / (ms * 1e-3), "form": ocd.kernel_form(p, B),
                             "frac_of_nominal_fp32": round(fl * B / (ms * 1e-3) / nominal, 4), "finite": finite})
    return rows


def cmaes_dropin_leg():
    """The same generation of BASELINE configs[1] end to end through the reference-facing drop-in: numpy candidates into
    `MPC_ORD.eval_weights_batch`, numpy returns out (host wall clock around the call: struct packing, the copy-in /
    kernel / copy-out graph of `ocd_episode_batch_host`, the synchronisation), and a short `optimize_cmaes` run with
    the CMA-ES bookkeeping between the generations."""
    import torch
    from l4dc_mpc_ocd_b200.interact_drive.reward_design.mpc_ord import MPC_ORD, finite_horizon_env
    car, world, inits = finite_horizon_env(horizon=5, env_seeds=[1, 2, 3, 4, 5], debug=False)
    ord_ = MPC_ORD(world, car, inits, designer_horizon=15, verbose=False)
    rng = np.random.default_rng(0)
    W = np.asarray(car.weights)[None] + 0.05 * rng.normal(size=(9, 7))
    for _ in range(5):
        ord_.eval_weights_batch(W)
    torch.cuda.synchronize()
    reps = 50
    t0 = time.perf_counter()
    for _ in range(reps):
        ord_.eval_weights_batch(W)
    ms = 1e3 * (time.perf_counter() - t0) / reps
    gens = 30
    t0 = time.perf_counter()
    ord_.optimize_cmaes(seed=1, sigma0=0.05, maxiter=gens)
    ms_opt = 1e3 * (time.perf_counter() - t0) / gens
    return {"workload": "finite_horizon cmaes --n_inits 5 through MPC_ORD (numpy in, numpy out): 9 candidates x 5 inits x 15 "
                        "control steps per generation",
            "eval_weights_batch_ms": ms, "candidate_evals_per_sec": 9 / (ms * 1e-3),
            "optimize_cmaes_ms_per_generation": ms_opt, "generations": gens}


def cmaes_multi_dropin_leg(world_size, max_over_ranks, barrier, runs_per_gpu=64, gens=60):
    """`cmaes_multi` end to end: `optimize_cmaes_lockstep` over 64 independent finite_horizon runs per GPU (n_inits 5
    each), host wall clock per generation -- the launch AND the Python side of a generation (CMA-ES updates of all runs
    as stacked numpy calls, candidate normalisation, per-run histories).  With N ranks the RUNS are spread over the
    ranks (`shard_runs=True`: rank k optimises runs k, k + N, ... on its own GPU, no collective until the results are
    exchanged at the end, which is inside the timed region)."""
    import torch
    from l4dc_mpc_ocd_b200.interact_drive.reward_design.mpc_ord import MPC_ORD, finite_horizon_env, optimize_cmaes_lockstep
    runs = runs_per_gpu * world_size

    def make():
        out = []
        for r in range(runs):
            car, world, inits = finite_horizon_env(horizon=5, env_seeds=[1000 + 5 * r + i for i in range(5)], debug=False)
            out.append(MPC_ORD(world, car, inits, designer_horizon=15, verbose=False))
        return out
    seeds = list(range(1, runs + 1))
    optimize_cmaes_lockstep(make(), seeds, sigma0=0.05, shard_runs=True, maxiter=2)      # graph capture, buffers
    rs = make()
    torch.cuda.synchronize()
    barrier()
    stats = {}
    t0 = time.perf_counter()
    optimize_cmaes_lockstep(rs, seeds, sigma0=0.05, shard_runs=True, stats=stats, maxiter=gens)
    dt = max_over_ranks(time.perf_counter() - t0)
    opt, exch = max_over_ranks(stats["optimise_s"]), max_over_ranks(stats["exchange_s"])
    return {"workload": f"finite_horizon cmaes --n_inits 5, {runs} independent runs ({runs_per_gpu} per GPU, spread over the "
                        f"ranks) in lock step through optimize_cmaes_lockstep, {gens} generations (+ the evaluation of "
                        f"the designer weights)",
            "ms_per_generation": 1e3 * dt / (gens + 1), "candidate_evals_per_sec": runs * (9 * gens + 1) / dt, "runs": runs,
            "optimise_ms_per_generation": 1e3 * opt / (gens + 1),
            "exchange_ms_once": 1e3 * exch,
            "note": "the value includes the one exchange of histories / results / object state at the end of the "
                    "optimisation (pickled all-gather; zero on one GPU), which a longer run amortises further"}


def cmaes_leg(eng, ocd, dist, rank, world_size, max_over_ranks, barrier, scenario, n_inits, runs=1):
    """BASELINE configs[1..3]: one CMA-ES generation of `run_mpc_ord.py <scenario> cmaes --n_inits n` = popsize 9
    candidates x n_inits initial states x samples episodes of T control steps, evaluated by ONE ocd_episode_batch
    launch; with N ranks the episodes are sharded and the per-episode returns all-gathered (NCCL).
    runs > 1: that many INDEPENDENT CMA-ES runs (different init groups, `--one_by_one` / the n_inits x seeds study of
    generalization_data.py) advanced in lock step -- their generations share the launch."""
    import torch
    from l4dc_mpc_ocd_b200.batched import compile_world, unlucky_sequence
    from l4dc_mpc_ocd_b200.experiments import run_mpc_ord
    env = run_mpc_ord.envs[scenario]
    T, ns = env["eval_horizon"], env["num_eval_samples"]
    car, world, inits = env["make_env"](env_seeds=[(1000000 + i) % (2 ** 32) for i in range(n_inits * runs)], debug=False)
    prog = compile_world(world, car)
    p, sc = prog.params, prog.scenario
    pop = 9                                               # pycma: 4 + floor(3 ln K), K = 7 or 6
    rng = np.random.default_rng(2024)
    w_true = np.asarray(car.weights, np.float64)
    w_true = (w_true / np.linalg.norm(w_true)).astype(np.float32)
    cand = w_true[None] + 0.05 * rng.normal(size=(runs * pop, p.K))
    cand = (cand / np.linalg.norm(cand, axis=1, keepdims=True)).astype(np.float32)
    I = np.asarray(inits, np.float32).reshape(runs, n_inits, 4)
    # episode (run r, candidate c, init i, sample s), flattened in that order
    ri = np.repeat(np.tile(I[:, None], (1, pop, 1, 1)).reshape(-1, 4), ns, axis=0)
    widx = np.repeat(np.arange(runs * pop, dtype=np.int32), n_inits * ns)
    B = ri.shape[0]
    ul = np.asarray(unlucky_sequence(world, B), np.int32) if prog.replanning else None
    per = (B + world_size - 1) // world_size
    dev = eng.device
    sel = np.minimum(np.arange(rank * per, rank * per + per), B - 1)     # shard padded to `per` episodes: regular all-gather
    ris = torch.as_tensor(np.ascontiguousarray(ri[sel].T), device=dev)
    w = torch.as_tensor(np.ascontiguousarray(cand.T), device=dev)
    idx = torch.as_tensor(widx[sel], device=dev)
    uls = None if ul is None else torch.as_tensor(ul[sel], device=dev)
    tw = torch.as_tensor(w_true, device=dev)
    out = dict(returns=torch.empty((per,), dtype=torch.float32, device=dev))
    gathered = torch.empty((per * world_size,), dtype=torch.float32, device=dev)

    def generation():
        eng.episodes_soa(p, sc, ris, w, runs * pop, tw, T, weight_idx=idx, unlucky_idx=uls, out=out)
        if dist is not None:
            dist.all_gather_into_tensor(gathered, out["returns"])
        else:
            gathered.copy_(out["returns"])
        return gathered[:B].reshape(runs * pop, n_inits * ns).sum(1) / ns

    for _ in range(3):
        generation()
    barrier()
    reps = 10
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        cand_returns = generation()
    e1.record()
    barrier()
    ms = max_over_ranks(float(e0.elapsed_time(e1))) / reps
    return {"workload": f"{scenario} cmaes --n_inits {n_inits}: one generation = {runs} run(s) x 9 candidates x {n_inits} inits x "
                        f"{ns} sample(s) x {T} control steps",
            "candidate_evals_per_sec": runs * pop / (ms * 1e-3), "ms_per_generation": ms, "runs": runs,
            "mpc_solves_per_generation": B * T, "episodes_per_rank": per, "kernel_form": ocd.kernel_form(p, per, True),
            "collective": "all_gather of per-episode returns (NCCL)" if dist is not None else "none (1 GPU)",
            "first_candidate_return": float(cand_returns[0].item())}


if __name__ == "__main__":
    main()
