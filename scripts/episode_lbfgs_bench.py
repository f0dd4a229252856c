"""Cost of receding-horizon episodes with the L-BFGS planner (ocd_episode_batch, optimizer 1) against the SGD episode,
of their implicit-function reverse pass (ocd_episode_implicit_vjp_batch) against the L-BFGS forward and the SGD
episodes_vjp, the rates of steps that hold controls and of singular steps, and a short Adam ascent on
MPC_ORD.eval_weights_grad with the L-BFGS planner.

    python scripts/episode_lbfgs_bench.py [--batches 4096,65536] [--warmup 1] [--reps 3] [--adam-steps 15]

Configurations: finite_horizon and replanning as `run_mpc_ord.py <scenario> cmaes --n_inits 5` evaluates one
generation (9 candidates x 5 initial states x num_eval_samples: 45 / 90 worlds of 15 / 20 control steps), and the
finite_horizon episode at the given batch sizes.  Each call is timed with CUDA events after warm-up: the SGD episode
(the scenario's math mode, fast) and the L-BFGS episode (precise: it has one form), both traced, then
episodes_implicit_vjp on the L-BFGS trace and episodes_vjp on the SGD trace (Engine.*_soa, workspace allocation
included, from the torch caching allocator after warm-up).  The status of every (world, step) of the implicit pass
gives the fractions of steps that hold controls at their value and of singular steps.  The GPU's name and power limit are read
in the same run.  The ascent runs Adam on eval_weights_grad from the designer weights on finite_horizon (5 initial
states) with the L-BFGS planner and prints the true return per step; it asserts nothing.  Prints only; writes no file.
"""
from __future__ import annotations

import argparse
import dataclasses
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "scripts"))

import l4dc_mpc_ocd_b200 as ocd                  # noqa: E402
import oracle as O                               # noqa: E402
from episode_vjp_bench import _params, gpu_info, time_ms    # noqa: E402


def bench(name: str, B: int, warmup: int, reps: int) -> str:
    spec = O.scenario_params(name)
    p, sc = _params(spec)
    pl = dataclasses.replace(p, optimizer=ocd.OPT_LBFGS, math_mode=ocd.MATH_PRECISE)
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
    tr = {q.optimizer: eng.episodes_soa(q, sc, ris, w, nc, tw, T, weight_idx=idx, unlucky_idx=ul, trace=True)
          for q in (p, pl)}
    rb = torch.ones((B,), device=dev)
    st = eng.episodes_implicit_vjp_soa(pl, sc, w, nc, tw, T, tr[1]["states"], tr[1]["best"], tr[1]["controls"], rb,
                                       idx, details=True)["status"].cpu().numpy()

    def fwd(q):
        return lambda: eng.episodes_soa(q, sc, ris, w, nc, tw, T, weight_idx=idx, unlucky_idx=ul, trace=True)

    def ivjp():
        eng.episodes_implicit_vjp_soa(pl, sc, w, nc, tw, T, tr[1]["states"], tr[1]["best"], tr[1]["controls"], rb,
                                      idx)

    def svjp():
        eng.episodes_vjp_soa(p, sc, w, nc, tw, T, tr[0]["states"], tr[0]["best"], tr[0]["controls"], rb, idx)
    ts, tl, ti, tv = (time_ms(f, warmup, reps) for f in (fwd(p), fwd(pl), ivjp, svjp))
    return (f"{name:14s} B {B:6d} T {T:2d}: SGD episode {ts:8.3f} ms   L-BFGS episode {tl:8.3f} ms   "
            f"implicit vjp {ti:8.3f} ms   SGD episodes_vjp {tv:8.3f} ms   "
            f"steps holding controls {np.mean(st > 0):6.1%}  singular {np.mean(st < 0):6.2%}")


def adam(steps: int, lr: float) -> None:
    from l4dc_mpc_ocd_b200.experiments import run_mpc_ord
    from l4dc_mpc_ocd_b200.interact_drive.reward_design.mpc_ord import MPC_ORD
    env = run_mpc_ord.envs["finite_horizon"]
    car, world, inits = env["make_env"](env_seeds=[1000000 + i for i in range(5)], debug=False)
    m = MPC_ORD(world, car, inits, env["eval_horizon"], num_samples=env["num_eval_samples"], verbose=False,
                planner_optimizer=ocd.OPT_LBFGS)
    x = np.array(m.designer_weights, dtype=np.float64)
    mom, vel = np.zeros_like(x), np.zeros_like(x)
    b1, b2, eps = 0.9, 0.999, 1e-8
    print(f"Adam on eval_weights_grad with the L-BFGS planner, finite_horizon, 5 initial states, lr {lr}")
    for it in range(steps + 1):
        obj, g = m.eval_weights_grad(x)
        print(f"step {it:3d}: true return {-obj:.5f}   |grad| {np.linalg.norm(g):.3e}")
        if it == steps or not np.isfinite(g).all():
            break
        mom = b1 * mom + (1 - b1) * g
        vel = b2 * vel + (1 - b2) * g * g
        x = x - lr * (mom / (1 - b1 ** (it + 1))) / (np.sqrt(vel / (1 - b2 ** (it + 1))) + eps)


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--batches", default="4096,65536")
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--adam-steps", type=int, default=15)
    ap.add_argument("--adam-lr", type=float, default=0.03)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("episode_lbfgs_bench needs a CUDA device (the engine has no CPU fallback)")
    print(f"device: {gpu_info()}")
    print(f"CUDA events, {a.warmup} warm-up + {a.reps} timed calls each")
    for name, B in [("finite_horizon", 45), ("replanning", 90)] + [("finite_horizon", int(x)) for x in a.batches.split(",")]:
        print(bench(name, B, a.warmup, a.reps), flush=True)
    adam(a.adam_steps, a.adam_lr)


if __name__ == "__main__":
    main()
