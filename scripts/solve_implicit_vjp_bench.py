"""Cost of the implicit-function VJP of the L-BFGS plan (ocd_solve_implicit_vjp_batch) against the L-BFGS forward solve
and against the unrolled VJP of the SGD solve (ocd_solve_vjp_batch) at the same shape.

    python scripts/solve_implicit_vjp_bench.py [--batches 256,4096,65536] [--warmup 2] [--reps 5]

Two shapes: finite_horizon (H 5, two cars, three lanes) and H 16 (the L-BFGS kernel's longest horizon), 100 iterations
each.  The L-BFGS solve and the implicit VJP run in precise math (the only math the L-BFGS kernel has); the SGD forward
and VJP in fast math, as the planner runs by default.  CUDA events around `reps` launches after `warmup` launches of
every kernel, the GPU's name and power limit read in the same run.  It also prints the share of problems whose reduced
Hessian was singular (NaN rows) and the median stationarity residual of the L-BFGS plans.  Prints only; writes no file.
"""
from __future__ import annotations

import argparse
import ctypes as C
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import l4dc_mpc_ocd_b200 as ocd                  # noqa: E402
from l4dc_mpc_ocd_b200 import synthetic          # noqa: E402

N = ocd._native


def gpu_info() -> str:
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        pl = "unknown"
    return f"{name}, power limit {pl or 'unknown'}"


def time_ms(fn, warmup: int, reps: int) -> float:
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(reps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / reps


def bench(H: int, lr_sgd: float, B: int, warmup: int, reps: int) -> dict:
    lb = ocd.PlannerParams(H=H, optimizer=ocd.OPT_LBFGS, math_mode=ocd.MATH_PRECISE)
    sgd = ocd.PlannerParams(H=H, lr=lr_sgd)
    dev = torch.device("cuda", 0)
    batch = synthetic.make_batch(B, seed=B + H)
    world = torch.as_tensor(batch["world"], device=dev).permute(1, 2, 0).contiguous()
    w = torch.as_tensor(batch["weights"], device=dev).t().contiguous()
    idx = torch.as_tensor(batch["weight_idx"], device=dev)
    ptr = lambda t: C.c_void_p(t.data_ptr())
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    pb = torch.randn((H, 2, B), device=dev)
    wbar, xbar, res = torch.empty((lb.K, B), device=dev), torch.empty((lb.C, 4, B), device=dev), torch.empty(B, device=dev)
    o_lb = dict(plan=torch.empty((H, 2, B), device=dev), losses=torch.empty((lb.S, B), device=dev),
                best=torch.empty((B,), dtype=torch.int32, device=dev))
    o_sgd = {k: torch.empty_like(v) for k, v in o_lb.items()}
    p_lb, p_sgd = lb.c_struct(), sgd.c_struct()
    nb = C.c_size_t(0)
    N.check(N.lib.ocd_solve_vjp_workspace_bytes(C.addressof(p_sgd), B, C.byref(nb)))
    ws = torch.empty((nb.value // 4,), device=dev)

    def solve(ps, o):
        N.check(N.lib.ocd_solve_batch(C.addressof(ps), ptr(world), None, 0, ptr(w), w.shape[1], ptr(idx), None,
                                      ptr(o["plan"]), ptr(o["losses"]), ptr(o["best"]), None, B, stream))

    def implicit():
        N.check(N.lib.ocd_solve_implicit_vjp_batch(C.addressof(p_lb), ptr(world), None, 0, ptr(w), w.shape[1],
                                                   ptr(idx), ptr(o_lb["plan"]), ptr(pb), ptr(wbar), ptr(xbar),
                                                   ptr(res), B, stream))

    def unrolled():
        N.check(N.lib.ocd_solve_vjp_batch(C.addressof(p_sgd), ptr(world), None, 0, ptr(w), w.shape[1], ptr(idx),
                                          None, ptr(o_sgd["best"]), ptr(pb), ptr(wbar), ptr(xbar), ptr(ws), nb.value,
                                          B, stream))
    solve(p_lb, o_lb)
    solve(p_sgd, o_sgd)
    out = dict(lbfgs=time_ms(lambda: solve(p_lb, o_lb), warmup, reps), implicit=time_ms(implicit, warmup, reps),
               sgd=time_ms(lambda: solve(p_sgd, o_sgd), warmup, reps), sgd_vjp=time_ms(unrolled, warmup, reps))
    implicit()
    torch.cuda.synchronize()
    out["singular"] = float(torch.isnan(wbar).any(0).float().mean())
    out["residual"] = float(res.median())
    return out


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--batches", default="256,4096,65536")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("solve_implicit_vjp_bench needs a CUDA device (the engine has no CPU fallback)")
    print(f"device: {gpu_info()}")
    print(f"C 2, L 3, n_iter 100; CUDA events, {a.warmup} warm-up + {a.reps} timed launches each")
    for H, lr_sgd in ((5, 0.1), (16, 0.02)):
        for B in (int(x) for x in a.batches.split(",")):
            r = bench(H, lr_sgd, B, a.warmup, a.reps)
            print(f"H {H:2d} B {B:6d}: lbfgs solve {r['lbfgs']:8.3f} ms  implicit_vjp {r['implicit']:8.3f} ms "
                  f"(x{r['implicit'] / r['lbfgs']:5.2f} of the solve) | sgd solve {r['sgd']:7.3f} ms  "
                  f"solve_vjp {r['sgd_vjp']:8.3f} ms | singular {100 * r['singular']:.1f} %, "
                  f"median residual {r['residual']:.1e}")


if __name__ == "__main__":
    main()
