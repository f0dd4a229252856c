"""Cost of the reverse pass through whole episodes (ocd_episode_vjp_batch) against the forward episode
(ocd_episode_batch) and against the sequential alternative -- T per-step solve VJPs -- and a short Adam ascent on
MPC_ORD.eval_weights_grad.

    python scripts/episode_vjp_bench.py [--batches 4096,65536] [--warmup 2] [--reps 5] [--adam-steps 25]

Configurations: finite_horizon and replanning as `run_mpc_ord.py <scenario> cmaes --n_inits 5` evaluates one
generation (9 candidates x 5 initial states x num_eval_samples: 45 / 90 worlds of 15 / 20 control steps), and the
finite_horizon episode at the given batch sizes.  Each is timed with CUDA events after warm-up: the forward episode
(without and with its trace), episodes_vjp (Engine.episodes_vjp_soa, workspace allocation included, from the torch
caching allocator after warm-up) and the sequential composition of T solve VJPs (Engine.solve_vjp_soa on each step's
traced world, one VJP per step; the host-side chain between them is not counted, so this is a lower bound of that
route).  The GPU's name and power limit are read in the same run.  The ascent runs Adam on eval_weights_grad from the
designer weights on finite_horizon (5 initial states) and prints the true return per step next to that of the
scenario's CMA-ES-tuned weights; it asserts nothing.  Prints only; writes no file.
"""
from __future__ import annotations

import argparse
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import l4dc_mpc_ocd_b200 as ocd                  # noqa: E402
import oracle as O                               # noqa: E402


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


def _params(spec) -> tuple:
    op, s = spec.params, spec.scenario
    p = ocd.PlannerParams(H=op.H, C=op.C, lane_x=tuple(op.lane_x), n_iter=op.n_iter, num_lanes=op.num_lanes,
                          other_mode=op.other_mode, extra_inits=op.extra_inits, lr=op.lr, dt=op.dt,
                          friction=op.friction, target_speed=op.target_speed)
    sc = ocd.Scenario(init_state=s.init_state, kind=s.kind, friction=s.friction, control=s.control, plan=s.plan,
                      critical_t=s.critical_t, teleport_state=s.teleport_state)
    return p, sc


def bench(name: str, B: int, warmup: int, reps: int) -> str:
    spec = O.scenario_params(name)
    p, sc = _params(spec)
    T = spec.eval_horizon
    eng = ocd.Engine(0)
    dev = eng.device
    rng = np.random.default_rng(B)
    ri = np.tile(spec.example_init.astype(np.float32), (B, 1))
    ri[:, 0] += rng.uniform(-0.03, 0.03, B).astype(np.float32)
    ri[:, 1] += rng.uniform(-0.04, 0.04, B).astype(np.float32)
    ri[:, 2] += rng.uniform(-0.08, 0.08, B).astype(np.float32)
    wt = (spec.designer_weights / np.linalg.norm(spec.designer_weights)).astype(np.float32)
    nc = 9
    cand = wt[None] + 0.05 * rng.normal(size=(nc, p.K))
    cand = (cand / np.linalg.norm(cand, axis=1, keepdims=True)).astype(np.float32)
    ris = torch.as_tensor(ri.T.copy(), device=dev)
    w = torch.as_tensor(cand.T.copy(), device=dev)
    tw = torch.as_tensor(wt, device=dev)
    idx = torch.as_tensor((np.arange(B) // max(1, B // nc)).clip(0, nc - 1).astype(np.int32), device=dev)
    ul = torch.as_tensor(rng.integers(1, p.C, B).astype(np.int32), device=dev) if spec.scenario.critical_t else None
    oc = None
    if p.other_mode == 1:       # the planner's model of the scripted cars in an episode, as solve_vjp's other_controls
        a = np.zeros((p.C - 1, p.H, 2, 1), np.float32)
        for j in range(p.C - 1):
            if spec.scenario.kind[j] == 1:
                for t in range(p.H):
                    pl = spec.scenario.plan[j]
                    a[j, t, :, 0] = pl[t] if t < len(pl) else spec.scenario.control[j]
        oc = torch.as_tensor(a, device=dev)
    tr = eng.episodes_soa(p, sc, ris, w, nc, tw, T, weight_idx=idx, unlucky_idx=ul, trace=True)
    rb = torch.ones((B,), device=dev)
    pb = torch.zeros((p.H, 2, B), device=dev)
    pb[0] = torch.randn((2, B), device=dev)

    def fwd():
        eng.episodes_soa(p, sc, ris, w, nc, tw, T, weight_idx=idx, unlucky_idx=ul)

    def fwd_trace():
        eng.episodes_soa(p, sc, ris, w, nc, tw, T, weight_idx=idx, unlucky_idx=ul, trace=True)

    def vjp():
        eng.episodes_vjp_soa(p, sc, w, nc, tw, T, tr["states"], tr["best"], tr["controls"], rb, idx)

    def seq():
        for t in range(T):
            eng.solve_vjp_soa(p, tr["states"][t], w, nc, tr["best"][t], pb, idx, oc, 1 if oc is not None else 0,
                              world_bar=True)
    tf, tt, tv, ts = (time_ms(f, warmup, reps) for f in (fwd, fwd_trace, vjp, seq))
    return (f"{name:14s} B {B:6d} T {T:2d}: episode {tf:8.3f} ms  (traced {tt:8.3f})   episodes_vjp {tv:8.3f} ms   "
            f"{T} x solve_vjp {ts:8.3f} ms   vjp / episode {tv / tf:5.1f}   sequential / vjp {ts / tv:5.2f}")


def adam(steps: int, lr: float) -> None:
    from l4dc_mpc_ocd_b200.experiments import run_mpc_ord
    from l4dc_mpc_ocd_b200.interact_drive.reward_design.mpc_ord import MPC_ORD
    env = run_mpc_ord.envs["finite_horizon"]
    car, world, inits = env["make_env"](env_seeds=[1000000 + i for i in range(5)], debug=False)
    m = MPC_ORD(world, car, inits, env["eval_horizon"], num_samples=env["num_eval_samples"], verbose=False)
    tuned = -m.eval_weights(O.scenario_params("finite_horizon").tuned_weights)
    x = np.array(m.designer_weights, dtype=np.float64)
    mom, vel = np.zeros_like(x), np.zeros_like(x)
    b1, b2, eps = 0.9, 0.999, 1e-8
    print(f"Adam on eval_weights_grad, finite_horizon, 5 initial states, lr {lr}; "
          f"return of the CMA-ES-tuned weights: {tuned:.5f}")
    for it in range(steps + 1):
        obj, g = m.eval_weights_grad(x)
        print(f"step {it:3d}: true return {-obj:.5f}   (tuned {tuned:.5f})   |grad| {np.linalg.norm(g):.3e}")
        if it == steps:
            break
        mom = b1 * mom + (1 - b1) * g
        vel = b2 * vel + (1 - b2) * g * g
        x = x - lr * (mom / (1 - b1 ** (it + 1))) / (np.sqrt(vel / (1 - b2 ** (it + 1))) + eps)


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--batches", default="4096,65536")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--adam-steps", type=int, default=25)
    ap.add_argument("--adam-lr", type=float, default=0.03)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("episode_vjp_bench needs a CUDA device (the engine has no CPU fallback)")
    print(f"device: {gpu_info()}")
    print(f"fast math; CUDA events, {a.warmup} warm-up + {a.reps} timed calls each")
    for name, B in [("finite_horizon", 45), ("replanning", 90)] + [("finite_horizon", int(x)) for x in a.batches.split(",")]:
        print(bench(name, B, a.warmup, a.reps), flush=True)
    adam(a.adam_steps, a.adam_lr)


if __name__ == "__main__":
    main()
