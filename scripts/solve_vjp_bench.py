"""Cost of the reverse pass through the solve (ocd_solve_vjp_batch) against the forward solve (ocd_solve_batch), and a
short plan-matching fit through torch.ops.ocd_b200.solve's autograd formula.

    python scripts/solve_vjp_bench.py [--batches 256,4096,65536] [--warmup 3] [--reps 10] [--fit-steps 60]

Times both kernels with CUDA events at the finite_horizon shape (H 5, two cars, three lanes, 100 SGD iterations, fast
math), after warm-up, and prints the times, their ratio and the GPU's name and power limit read in the same run.  The fit
plants a weight vector, takes its plans on 256 problems as the target and runs Adam on a normalised weight vector from a
perturbed start; it reports what happened and asserts nothing.  Prints only; writes no file.
"""
from __future__ import annotations

import argparse
import ctypes as C
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import l4dc_mpc_ocd_b200 as ocd                  # noqa: E402
from l4dc_mpc_ocd_b200 import synthetic          # noqa: E402
from l4dc_mpc_ocd_b200 import torch_ops as T     # noqa: E402

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


def bench(B: int, warmup: int, reps: int) -> tuple[float, float]:
    p = ocd.PlannerParams()                          # finite_horizon: H 5, C 2, lanes (-0.1, 0, 0.1), 100 iterations
    eng = ocd.Engine(0)
    dev = eng.device
    batch = synthetic.make_batch(B, seed=B)
    world = torch.as_tensor(batch["world"], device=dev).permute(1, 2, 0).contiguous()
    w = torch.as_tensor(batch["weights"], device=dev).t().contiguous()
    idx = torch.as_tensor(batch["weight_idx"], device=dev)
    out = dict(plan=torch.empty((p.H, 2, B), device=dev), losses=torch.empty((p.S, B), device=dev),
               best=torch.empty((B,), dtype=torch.int32, device=dev))
    eng.solve_soa(p, world, w, w.shape[1], idx, out=out)
    ps = p.c_struct()
    nb = C.c_size_t(0)
    N.check(N.lib.ocd_solve_vjp_workspace_bytes(C.addressof(ps), B, C.byref(nb)))
    ws = torch.empty((nb.value // 4,), device=dev)
    pb = torch.randn((p.H, 2, B), device=dev)
    wbar, xbar = torch.empty((p.K, B), device=dev), torch.empty((p.C, 4, B), device=dev)
    ptr = lambda t: C.c_void_p(t.data_ptr())
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def fwd():
        N.check(N.lib.ocd_solve_batch(C.addressof(ps), ptr(world), None, 0, ptr(w), w.shape[1], ptr(idx), None,
                                      ptr(out["plan"]), ptr(out["losses"]), ptr(out["best"]), None, B, stream))

    def vjp():
        N.check(N.lib.ocd_solve_vjp_batch(C.addressof(ps), ptr(world), None, 0, ptr(w), w.shape[1], ptr(idx), None,
                                          ptr(out["best"]), ptr(pb), ptr(wbar), ptr(xbar), ptr(ws), nb.value, B, stream))
    return time_ms(fwd, warmup, reps), time_ms(vjp, warmup, reps)


def fit(steps: int) -> None:
    p = ocd.PlannerParams()
    dev = torch.device("cuda", 0)
    B = 256
    batch = synthetic.make_batch(B, seed=77)
    world = torch.as_tensor(batch["world"], device=dev).permute(1, 2, 0).contiguous()
    rng = np.random.default_rng(5)
    w_true = rng.normal(size=p.K)
    w_true /= np.linalg.norm(w_true)
    wt = torch.as_tensor(w_true[:, None], dtype=torch.float32, device=dev)
    with torch.no_grad():
        target = torch.ops.ocd_b200.solve(world, wt, None, None, T.pack_params(p))[0]
    v = torch.as_tensor((w_true + 0.4 * rng.normal(size=p.K))[:, None], dtype=torch.float32, device=dev)
    v.requires_grad_(True)
    opt = torch.optim.Adam([v], lr=0.02)
    for it in range(steps + 1):
        w = v / v.norm()
        plan = torch.ops.ocd_b200.solve(world, w, None, None, T.pack_params(p))[0]
        loss = ((plan - target) ** 2).mean()
        if it % 10 == 0 or it == steps:
            cos = float((w.detach()[:, 0].double().cpu().numpy() @ w_true))
            print(f"fit step {it:3d}: plan-matching loss {loss.item():.3e}, cos(w, w_planted) {cos:.4f}")
        if it == steps:
            break
        opt.zero_grad()
        loss.backward()
        opt.step()


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--batches", default="256,4096,65536")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--fit-steps", type=int, default=60)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("solve_vjp_bench needs a CUDA device (the engine has no CPU fallback)")
    print(f"device: {gpu_info()}")
    print("finite_horizon shape: H 5, C 2, L 3, n_iter 100, fast math; CUDA events, "
          f"{a.warmup} warm-up + {a.reps} timed launches each")
    for B in (int(x) for x in a.batches.split(",")):
        tf, tv = bench(B, a.warmup, a.reps)
        print(f"B {B:6d}: solve {tf:8.3f} ms   solve_vjp {tv:8.3f} ms   ratio {tv / tf:6.1f}")
    fit(a.fit_steps)


if __name__ == "__main__":
    main()
