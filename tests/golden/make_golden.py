#!/usr/bin/env python
"""Generate the golden vectors in tests/golden/*.json from the REFERENCE'S OWN PYTHON.

Needs a checkout of the reference (avikj/L4DC-MPC-OCD), which is not part of this repository:
pass it as --reference DIR or in L4DC_REFERENCE_DIR.  The tests only read the committed JSON
files.  The reference modules are imported unmodified from that checkout; the TensorFlow
primitives they call are supplied by the torch-backed stand-in in oracle/tf_shim (see
oracle/ocd_oracle.h "PARITY STATUS").  Nothing from this repo's oracle or engine is used to
produce the numbers.

    python tests/golden/make_golden.py --reference DIR --all --jobs 8      # ~15 min on 8 cores
    python tests/golden/make_golden.py --reference DIR --part primitives   # one part

Parts: primitives, features, mpc_reward, plans, planner_kats, and one episode_* part per
(scenario, weights, variant).
"""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import time
from pathlib import Path

HERE = Path(__file__).resolve().parent
REPO = HERE.parent.parent


def _setup_reference_imports(ref: Path):
    if not (ref / "interact_drive").is_dir():
        raise SystemExit(f"make_golden.py needs a checkout of the reference: {ref} has no interact_drive/")
    sys.path.insert(0, str(REPO / "oracle" / "tf_shim"))
    sys.path.insert(0, str(ref))
    os.chdir(ref)  # the library imports the `experiments` package relative to the repo root


def _f(x):
    """JSON-safe float lists with full float32 precision."""
    import numpy as np
    a = np.asarray(x)
    if a.ndim == 0:
        return float(a)
    return [_f(e) for e in a]


@contextlib.contextmanager
def _quiet():
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        yield


# ---------------------------------------------------------------------------------------------
def part_primitives():
    import numpy as np
    import tensorflow as tf
    from interact_drive.math_utils import _f as ref_f, smooth_threshold, smooth_bump
    from interact_drive.simulation_utils import next_car_state

    out = {"source": "interact_drive/math_utils.py, interact_drive/simulation_utils.py on oracle/tf_shim"}
    # doctest points (math_utils.py:19-26, 65-71, 140-148)
    out["f_doctest"] = {"f(0)": _f(ref_f(tf.constant(0.)).numpy()), "f(1)": _f(ref_f(tf.constant(1.)).numpy()),
                        "f(0.01)": _f(ref_f(tf.constant(0.01)).numpy()), "f(1e10)": _f(ref_f(tf.constant(1e10)).numpy())}
    t = smooth_threshold(0., 1.)
    out["threshold_doctest"] = {k: _f(t(tf.constant(v)).numpy()) for k, v in (("0", 0.), ("-1", -1.), ("-0.5", -0.5))}
    b = smooth_bump(-1., 1.)
    out["bump_doctest"] = {k: _f(b(tf.constant(v)).numpy()) for k, v in (("0", 0.), ("-1", -1.), ("1", 1.), ("0.5", 0.5))}

    rng = np.random.default_rng(7)
    f_pts = []
    for x in list(rng.uniform(-0.02, 0.08, 12)) + [0.0, 1e-3, 0.05]:
        for shape in (5.0, 100.0):
            f_pts.append({"x": float(np.float32(x)), "shape": shape,
                          "y": _f(ref_f(tf.constant(np.float32(x)), tf.constant(shape)).numpy())})
    out["f"] = f_pts
    thr_pts = []
    for (thr, width) in ((0.15000000000000002, 0.05), (0.1, 0.05), (0.0, 1.0)):
        tfn = smooth_threshold(thr, width=width)
        lo, hi = thr - 1.6 * width, thr + 0.6 * width
        for z in list(rng.uniform(lo, hi, 14)) + [thr, thr - width, thr - width / 2]:
            thr_pts.append({"threshold": thr, "width": width, "z": float(np.float32(z)),
                            "y": _f(tfn(tf.constant(np.float32(z))).numpy())})
    out["threshold"] = thr_pts
    bump_pts = []
    for (c, w) in ((0.0, 0.08), (-0.6, 0.15), (0.1, 0.08), (-0.37, 0.15)):
        start = tf.constant(np.float32(c)) - w
        end = tf.constant(np.float32(c)) + w
        bfn = smooth_bump(start, end)
        for z in list(rng.uniform(c - 1.3 * w, c + 1.3 * w, 12)) + [c, c - w, c + w]:
            bump_pts.append({"start": _f(start.numpy()), "end": _f(end.numpy()), "z": float(np.float32(z)),
                             "y": _f(bfn(tf.constant(np.float32(z))).numpy())})
    out["bump"] = bump_pts

    dyn = []
    kat = [([0., 0., 1., np.pi / 2], [0., 0.], 1.0, 0.0), ([0., 0., 1., np.pi / 2], [0., 0.], 1.0, 1.0),
           ([0., 0., 1., np.pi / 2], [0., 0.], 1.0, 0.5), ([0., 0., 1., 0.], [0., 0.], 1.0, 0.5)]
    for s, u, dt, mu in kat:  # test_simulation_utils.py:113-158 (same numbers through next_car_state)
        dyn.append({"state": s, "control": u, "dt": dt, "friction": mu, "kat": True,
                    "next": _f(next_car_state(tf.constant(s, dtype=tf.float32), tf.constant(u, dtype=tf.float32), dt,
                                              tf.constant(mu)).numpy())})
    for _ in range(24):
        s = [rng.uniform(-0.2, 0.2), rng.uniform(-1, 1), rng.uniform(0, 1.5), rng.uniform(0, np.pi)]
        u = [rng.uniform(-10, 6), rng.uniform(-6, 6)]
        mu = float(rng.choice([0.0, 0.2, 0.5]))
        s32, u32 = [float(np.float32(v)) for v in s], [float(np.float32(v)) for v in u]
        dyn.append({"state": s32, "control": u32, "dt": 0.1, "friction": mu, "kat": False,
                    "next": _f(next_car_state(tf.constant(s32, dtype=tf.float32), tf.constant(u32, dtype=tf.float32),
                                              0.1, tf.constant(mu)).numpy())})
    out["dynamics"] = dyn
    return out


def _make_world(kind: str, n_other: int, rng, other_states=None):
    """Worlds built from the reference's classes (cars are placed explicitly)."""
    import numpy as np
    from interact_drive.world import ThreeLaneCarWorld, TwoLaneCarWorld
    from interact_drive.car import FixedVelocityCar
    from experiments.merging import ThreeLaneTestCar
    if kind == "three":
        world = ThreeLaneCarWorld()
        K, ts, nl = 7, 1.0, 3
    else:
        world = TwoLaneCarWorld()
        K, ts, nl = 6, 1.2, 2
    w = rng.normal(size=K)
    with _quiet():
        robot = ThreeLaneTestCar(world, np.array([0., -0.9, 0.8, np.pi / 2]), horizon=5, weights=w,
                                 target_speed=ts, num_lanes=nl)
    cars = [robot]
    for j in range(n_other):
        st = np.array([0., -0.6, 0.5, np.pi / 2]) if other_states is None else np.asarray(other_states[j])
        cars.append(FixedVelocityCar(world, st, horizon=5))
    world.add_cars(cars)
    world.reset()
    return world, robot


def _random_world_state(rng, n_other, kind, hard=False):
    import numpy as np
    half = 0.15 if kind == "three" else 0.1
    x = rng.uniform(-half - 0.04, half + 0.04)
    y = rng.uniform(-1.0, -0.6)
    v = rng.uniform(0.3, 1.4) if not hard else rng.uniform(-1.5, 3.5)
    th = np.pi / 2 + rng.uniform(-0.6, 0.6)
    st = [[x, y, v, th]]
    for _ in range(n_other):
        ox = float(rng.choice([-0.1, 0.0, 0.1, -0.05, 0.05])) + rng.uniform(-0.01, 0.01)
        oy = y + rng.uniform(-0.2, 0.3)
        st.append([ox, oy, rng.uniform(0.3, 1.0), np.pi / 2 + rng.uniform(-0.3, 0.3)])
    return np.asarray(st, dtype=np.float32)


def part_features():
    import numpy as np
    import tensorflow as tf
    rng = np.random.default_rng(11)
    cases = []
    for kind, n_other in (("three", 1), ("three", 2), ("two", 2), ("three", 4)):
        world, robot = _make_world(kind, n_other, rng)
        for i in range(16):
            st = _random_world_state(rng, n_other, kind, hard=(i % 5 == 4))
            if i == 0:   # exact lane tie / zero crossing points
                st[0, 0] = 0.05 if kind == "three" else 0.0
            if i == 1:
                st[0, 0] = 0.0
            if i == 2 and n_other >= 2:   # two cars at the same place: tie in the max
                st[2] = st[1]
                st[0, 0], st[0, 1] = st[1, 0] + 0.02, st[1, 1] - 0.05
            state = [tf.constant(r, dtype=tf.float32) for r in st]
            phi = robot.features(state, tf.constant([0., 0.]))
            cases.append({"world": kind, "lane_x": [float(l.p[0]) for l in world.lanes],
                          "num_lanes": int(robot.num_lanes), "target_speed": float(robot.target_speed),
                          "state": _f(st), "phi": _f(phi.numpy())})
    return {"source": "experiments/merging.py ThreeLaneTestCar.features on oracle/tf_shim", "cases": cases}


def part_mpc_reward():
    import numpy as np
    import tensorflow as tf
    from interact_drive.planner.naive_planner import NaivePlanner
    rng = np.random.default_rng(13)
    cases = []
    for kind, n_other, H, mode in (("three", 1, 5, 0), ("three", 1, 6, 0), ("two", 2, 5, 1), ("three", 3, 3, 0),
                                   ("three", 2, 8, 1), ("three", 1, 15, 0)):
        for rep in range(6):
            st = _random_world_state(rng, n_other, kind)
            st[0, 3] = np.pi / 2 + rng.uniform(-0.2, 0.2)
            world, robot = _make_world(kind, n_other, rng)
            with _quiet():
                planner = NaivePlanner(world, robot, horizon=H)
            init_state = [tf.constant(r, dtype=tf.float32) for r in st]
            scale = 1.0 if rep < 4 else 6.0     # rep 4,5: controls beyond the clip limits
            u_np = (rng.normal(size=(H, 2)) * np.array([1.0, 1.5]) * scale).astype(np.float32)
            controls = [tf.Variable(u, dtype=tf.float32) for u in u_np]
            oc_np = None
            other_controls = None
            if mode == 1:
                oc_np = (rng.normal(size=(n_other, H, 2)) * np.array([0.7, 2.0])).astype(np.float32)
                other_controls = [tf.constant(np.zeros((H, 1), np.float32))] + \
                                 [tf.constant(oc_np[j]) for j in range(n_other)]
            w = robot.weights
            with tf.GradientTape() as tape:
                R = planner.reward_func(init_state, controls, other_controls=other_controls)
            grads = tape.gradient(R, controls)
            cases.append({"world": kind, "lane_x": [float(l.p[0]) for l in world.lanes],
                          "num_lanes": int(robot.num_lanes), "target_speed": float(robot.target_speed),
                          "H": H, "other_mode": mode, "friction": float(robot.friction), "dt": float(world.dt),
                          "init_state": _f(st), "controls": _f(u_np),
                          "other_controls": None if oc_np is None else _f(oc_np),
                          "weights": _f(w), "R": _f(R.numpy()),
                          "grad": _f(np.stack([np.zeros(2, np.float32) if g is None else g.numpy() for g in grads]))})
    return {"source": "interact_drive/planner/naive_planner.py:32-79 mpc_reward + shim autograd", "cases": cases}


def _scenario(name, **kw):
    with _quiet():
        if name == "finite_horizon":
            from interact_drive.reward_design.mpc_ord import finite_horizon_env
            return finite_horizon_env(env_seeds=[1000000], debug=True, **kw)
        if name == "local_opt":
            from experiments.local_opt_scenario import local_opt_env
            return local_opt_env(env_seeds=[1000000], debug=True, **kw)
        if name == "replanning":
            from experiments.replanning_world import setup_world
            return setup_world(env_seeds=[1000000], debug=True, **kw)
    raise KeyError(name)


_TUNED = {   # experiments/run_mpc_ord.py:25-26,34-35,42
    "local_opt": [-0.09686739, 0.25720383, -0.58355971, -0.23075428, -0.41237239, -0.4758984, -0.36625558],
    "finite_horizon": [-0.21963165, -0.01184596, 0.34379187, -0.04687411, -0.06364365, -0.54138792, -0.7308079],
    "replanning": [-0.55899817, -0.4436692, -0.3724511, -0.19964276, -0.5438697, 0.12770043],
}
_EVAL = {"local_opt": (15, 1), "finite_horizon": (15, 1), "replanning": (20, 2)}   # run_mpc_ord.py:19-44


def part_plans():
    """generate_plan at the scenario's first control step, for several weight vectors."""
    import numpy as np
    rng = np.random.default_rng(17)
    cases = []
    for name in ("finite_horizon", "local_opt", "replanning"):
        car, world, inits = _scenario(name)
        K = len(car.weights)
        true_w = car.weights.copy()
        wsets = [("true", true_w), ("tuned", np.asarray(_TUNED[name])), ("random", rng.normal(size=K))]
        for label, w in wsets:
            car.weights = w
            import tensorflow as tf
            car.init_state = tf.constant(inits[0], dtype=tf.float32)
            world.reset()
            if name == "replanning":
                # the same call PlannerCar._get_next_control makes (planner_car.py:54-85)
                ctrl = car._get_next_control()
                plan = car.plan
            else:
                ctrl = car._get_next_control()
                plan = car.plan
            cases.append({"scenario": name, "weights_label": label, "weights_in": _f(w),
                          "weights_normalised": _f(car.weights), "init": _f(np.asarray(inits[0], np.float32)),
                          "world_state": _f(np.stack([s.numpy() if hasattr(s, "numpy") else np.asarray(s, np.float32)
                                                      for s in world.state])),
                          "plan": _f(np.stack([p.numpy() for p in plan])), "control": _f(ctrl.numpy())})
    return {"source": "PlannerCar._get_next_control -> NaivePlanner.generate_plan on oracle/tf_shim", "cases": cases}


def part_planner_kats():
    """interact_drive/planner/tests/test_naivePlanner.py:21-32 and :50-63, run as written."""
    import numpy as np
    from interact_drive.planner.naive_planner import NaivePlanner
    from interact_drive.world import ThreeLaneCarWorld
    from interact_drive.planner.tests.targetSpeedRewardMaximizerCar import TargetSpeedPlannerCar
    out = []
    for friction, horizon, n_iter in ((0.0, 5, 100), (0.5, 3, 500)):
        world = ThreeLaneCarWorld()
        init_state = np.array([0., 0., 1., np.pi / 2], dtype=np.float32)
        car = TargetSpeedPlannerCar(world, init_state, 4, target_speed=1., friction=friction)
        world.add_car(car)
        with _quiet():
            planner = NaivePlanner(world, car, horizon=horizon, learning_rate=5.0, n_iter=n_iter)
        plan = planner.generate_plan([car.state])
        out.append({"friction": friction, "horizon": horizon, "n_iter": n_iter, "learning_rate": 5.0,
                    "init_state": _f(init_state), "target_speed": 1.0,
                    "plan": _f(np.stack([p.numpy() for p in plan])),
                    "expected": [[friction * 1.0 ** 2, 0.0]] * horizon, "atol": 1e-5})
    return {"source": "interact_drive/planner/tests/test_naivePlanner.py on oracle/tf_shim", "cases": out}


def part_episode(name: str, wlabel: str, variant: str):
    """MPC_ORD.eval_weights_for_init (mpc_ord.py:67-106) with num_samples=1, once per outcome."""
    import numpy as np
    from interact_drive.reward_design.mpc_ord import MPC_ORD
    kw = {}
    if variant == "extra_inits":
        kw["extra_inits"] = True
    if variant == "h6":
        kw["horizon"] = 6
    car, world, inits = _scenario(name, **kw)
    T, nsamp = _EVAL[name]
    if variant == "short":
        T = 6
    w_in = car.weights.copy() if wlabel == "true" else np.asarray(_TUNED[name])
    if wlabel == "scaled":
        w_in = car.weights.copy() * 3.7    # exercises the triple normalisation (mpc_ord.py:71,120)
    m = MPC_ORD(world, car, inits, T, num_samples=1)
    samples = []
    for k in range(nsamp):
        t0 = time.time()
        with _quiet():
            r = m.eval_weights_for_init(inits[0], np.array(w_in, dtype=np.float64), False)
        traj = car.past_traj
        rec = {"return": _f(r), "seconds": time.time() - t0,
               "unlucky_car_idx": int(getattr(world, "unlucky_car_idx", 0)),
               "controls": _f(np.stack([c.numpy() for (_, c) in traj])),
               "robot_states": _f(np.stack([np.asarray(s.numpy() if hasattr(s, "numpy") else s, np.float32)
                                            for (s, _) in traj])),
               "other_states": [_f(np.stack([np.asarray(s.numpy() if hasattr(s, "numpy") else s, np.float32)
                                             for (s, _) in oc.past_traj])) for oc in world.cars[1:]]}
        samples.append(rec)
    return {"source": "MPC_ORD.eval_weights_for_init on oracle/tf_shim (reference code unmodified)",
            "scenario": name, "weights_label": wlabel, "variant": variant, "T": T,
            "weights_in": _f(w_in), "plan_weights": _f(car.weights), "true_weights": _f(m.designer_weights),
            "init": _f(np.asarray(inits[0])), "horizon": int(car.horizon),
            "n_iter": int(car.planner.n_iter), "extra_inits": bool(car.planner.extra_inits),
            "samples": samples}


EPISODES = [
    ("finite_horizon", "true", "full"), ("finite_horizon", "tuned", "full"),
    ("finite_horizon", "true", "extra_inits"), ("finite_horizon", "true", "h6"),
    ("local_opt", "true", "full"), ("local_opt", "tuned", "full"), ("local_opt", "scaled", "short"),
    ("local_opt", "true", "extra_inits"),
    ("replanning", "true", "full"), ("replanning", "tuned", "full"),
]
SIMPLE = {"primitives": part_primitives, "features": part_features, "mpc_reward": part_mpc_reward,
          "plans": part_plans, "planner_kats": part_planner_kats}


def run_part(part: str, ref: Path, outdir: Path = HERE):
    _setup_reference_imports(ref)
    t0 = time.time()
    if part in SIMPLE:
        data = SIMPLE[part]()
    else:
        _, name, wlabel, variant = part.split(":")
        data = part_episode(name, wlabel, variant)
    data["generated_by"] = "tests/golden/make_golden.py --part " + part
    data["generator_seconds"] = round(time.time() - t0, 1)
    fname = part.replace(":", "_") + ".json"
    with open(Path(outdir) / fname, "w") as f:
        json.dump(data, f, indent=1)
    print("wrote", fname, "in %.0fs" % (time.time() - t0), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--part")
    ap.add_argument("--all", action="store_true")
    ap.add_argument("--jobs", type=int, default=8)
    ap.add_argument("--outdir", default=str(HERE), help="where to write the JSON (default: tests/golden)")
    ap.add_argument("--reference", default=os.environ.get("L4DC_REFERENCE_DIR"),
                    help="checkout of the reference (default: $L4DC_REFERENCE_DIR)")
    args = ap.parse_args()
    if not args.reference:
        ap.error("--reference DIR (or L4DC_REFERENCE_DIR) must name a checkout of the reference")
    ref = Path(args.reference).resolve()
    parts = list(SIMPLE) + ["episode:%s:%s:%s" % e for e in EPISODES]
    if args.part:
        run_part(args.part, ref, Path(args.outdir).resolve())
        return
    if not args.all:
        ap.error("--part NAME or --all")
    pending, running = list(parts), []
    while pending or running:
        while pending and len(running) < args.jobs:
            p = pending.pop(0)
            running.append((p, subprocess.Popen([sys.executable, __file__, "--part", p, "--reference", str(ref)])))
        time.sleep(2)
        for item in list(running):
            if item[1].poll() is not None:
                running.remove(item)
                if item[1].returncode:
                    print("FAILED", item[0], flush=True)


if __name__ == "__main__":
    main()
