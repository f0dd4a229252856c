"""Pins the CPU oracle (oracle/: C restatement of the reference's planner path) against the golden
vectors produced by the reference's own unmodified Python (tests/golden/make_golden.py) and against
the reference's known-answer tests.  CPU only."""
import numpy as np
import pytest

import oracle as O
from l4dc_mpc_ocd_b200 import synthetic
from conftest import load_golden

F32 = np.float32


def _params(c, **kw):
    st = np.asarray(c.get("state", c.get("init_state")), F32)
    return O.OracleParams(C=st.shape[0], lane_x=tuple(c["lane_x"]), num_lanes=c["num_lanes"],
                          target_speed=c["target_speed"], **kw)


def test_dynamics_known_answers_and_golden():
    g = load_golden("primitives.json")
    for c in g["dynamics"]:
        out = O.dynamics_step(c["state"], c["control"], c["dt"], c["friction"])
        np.testing.assert_allclose(out, np.asarray(c["next"], F32), rtol=0, atol=1e-7)
    hp = np.pi / 2   # interact_drive/tests/test_simulation_utils.py:113-158
    np.testing.assert_allclose(O.dynamics_step([0, 0, 1, hp], [0, 0], 1.0, 0.0), [0, 1, 1, hp], atol=1e-6)
    np.testing.assert_allclose(O.dynamics_step([0, 0, 1, hp], [0, 0], 1.0, 1.0), [0, 0.5, 0, hp], atol=1e-6)
    np.testing.assert_allclose(O.dynamics_step([0, 0, 1, hp], [0, 0], 1.0, 0.5), [0, 0.75, 0.5, hp], atol=1e-6)
    np.testing.assert_allclose(O.dynamics_step([0, 0, 1, 0], [0, 0], 1.0, 0.5), [0.75, 0, 0.5, 0], atol=1e-6)


def test_smooth_helpers_doctests_and_golden():
    g = load_golden("primitives.json")
    assert O.smooth_f(0.0) == 0.0 and O.smooth_f(1.0) > 0 and abs(O.smooth_f(1e10) - 1) < 1e-7
    assert O.smooth_threshold(0.0, 0.0, 1.0) == 1.0 and O.smooth_threshold(-1.0, 0.0, 1.0) == 0.0
    assert abs(O.smooth_threshold(-0.5, 0.0, 1.0) - 0.5) < 1e-7
    assert O.smooth_bump(0.0, -1.0, 1.0) == 1.0 and O.smooth_bump(1.0, -1.0, 1.0) == 0.0 and \
        O.smooth_bump(-1.0, -1.0, 1.0) == 0.0 and O.smooth_bump(0.5, -1.0, 1.0) > 0
    for k, v in g["f_doctest"].items():
        assert abs(O.smooth_f(float(k[2:-1])) - v) <= 1e-7
    for c in g["f"]:
        assert abs(O.smooth_f(c["x"], c["shape"]) - c["y"]) <= 2e-7 * max(1, abs(c["y"]))
    for c in g["threshold"]:
        assert abs(O.smooth_threshold(c["z"], c["threshold"], c["width"]) - c["y"]) <= 5e-7
    for c in g["bump"]:
        assert abs(O.smooth_bump(c["z"], c["start"], c["end"]) - c["y"]) <= 5e-7


def test_features_golden():
    for c in load_golden("features.json")["cases"]:
        phi = O.features(_params(c), np.asarray(c["state"], F32))
        np.testing.assert_allclose(phi, np.asarray(c["phi"], F32), rtol=2e-6, atol=2e-7)


def test_mpc_reward_and_gradient_golden():
    """Value and d/d controls against the reference's mpc_reward under autograd."""
    for c in load_golden("mpc_reward.json")["cases"]:
        p = _params(c, H=c["H"], other_mode=c["other_mode"], friction=c["friction"], dt=c["dt"])
        R, G = O.mpc_reward(p, c["init_state"], c["controls"], c["weights"], other_controls=c["other_controls"])
        gref = np.asarray(c["grad"], F32)
        assert abs(R - c["R"]) <= 2e-6 * max(1.0, abs(c["R"]))
        assert np.max(np.abs(G - gref)) <= 2e-6 * max(1.0, np.abs(gref).max())


def test_adjoint_against_finite_differences_f64():
    rng = np.random.default_rng(3)
    for trial in range(40):
        C, H = int(rng.integers(2, 5)), int(rng.integers(3, 9))
        lanes = (-0.1, 0.0, 0.1) if trial % 2 else (-0.05, 0.05)
        p = O.OracleParams(H=H, C=C, lane_x=lanes, num_lanes=len(lanes), other_mode=trial % 3 == 0)
        world = np.zeros((C, 4))
        world[:, 0] = rng.uniform(-0.12, 0.12, C)
        world[:, 1] = rng.uniform(-1, -0.6, C)
        world[:, 2] = rng.uniform(0.4, 1.2, C)
        world[:, 3] = np.pi / 2 + rng.uniform(-0.3, 0.3, C)
        u = rng.normal(size=(H, 2)) * [1.0, 1.5]
        w = rng.normal(size=p.K)
        oc = rng.normal(size=(C - 1, H, 2)) if p.other_mode else None
        R, G = O.mpc_reward(p, world, u, w, other_controls=oc, dtype=np.float64)
        eps = 1e-6
        for (t, k) in ((0, 0), (H - 1, 1), (H // 2, 0), (H // 2, 1)):
            up, um = u.copy(), u.copy()
            up[t, k] += eps
            um[t, k] -= eps
            fd = (O.mpc_reward(p, world, up, w, other_controls=oc, dtype=np.float64, grad=False)
                  - O.mpc_reward(p, world, um, w, other_controls=oc, dtype=np.float64, grad=False)) / (2 * eps)
            assert abs(fd - G[t, k]) <= 1e-5 * max(1.0, abs(fd)), (trial, t, k, fd, G[t, k])


def test_clip_masks_follow_tensorflow():
    """d clip / d u = 1 on the closed interval (SURVEY A.3): at the bound the gradient passes,
    beyond it it is exactly zero."""
    p = O.OracleParams(H=3, C=2)
    world = np.array([[0.02, -0.9, 0.8, np.pi / 2], [0.0, -0.6, 0.5, np.pi / 2]], F32)
    w = np.array([-0.5, 0.1, 0.2, 0.3, -0.2, -0.5, -0.5], F32)
    u = np.array([[4.0, 4.0], [4.5, -4.5], [-8.0, -4.0]], F32)
    _, G = O.mpc_reward(p, world, u, w)
    assert G[1, 0] == 0 and G[1, 1] == 0
    assert G[0, 0] != 0 and G[2, 0] != 0 and G[2, 1] != 0


def test_planner_known_answers():
    """interact_drive/planner/tests/test_naivePlanner.py:21-32, :50-63 (atol 1e-5 there)."""
    for c in load_golden("planner_kats.json")["cases"]:
        p = O.OracleParams(H=c["horizon"], C=2, n_iter=c["n_iter"], lr=c["learning_rate"], friction=c["friction"])
        world = np.asarray([c["init_state"], [50.0, 50.0, 0.0, np.pi / 2]], F32)
        r = O.generate_plan(p, world, [-1, 0, 0, 0, 0, 0, 0])
        np.testing.assert_allclose(r["plan"], np.asarray(c["expected"]), atol=1e-5)
        np.testing.assert_allclose(r["plan"], np.asarray(c["plan"]), atol=1e-6)


def test_lbfgs_restatement_sanity():
    """The opt-in L-BFGS (params.optimizer == 1) has no running reference counterpart (naive_planner.py:127-149
    is dead code on an absent dependency) -- parity for it is UNPINNED.  What can be checked on the CPU twin: it
    reaches the reference's planner KATs, never ends a start above where it began (Armijo), and on random problems
    finds objectives at least as good as the reference's 100 SGD steps for the large majority."""
    from l4dc_mpc_ocd_b200 import synthetic
    for c in load_golden("planner_kats.json")["cases"]:
        p = O.OracleParams(H=c["horizon"], C=2, n_iter=200, lr=c["learning_rate"], friction=c["friction"], optimizer=1)
        world = np.asarray([c["init_state"], [50.0, 50.0, 0.0, np.pi / 2]], F32)
        r = O.generate_plan(p, world, [-1, 0, 0, 0, 0, 0, 0])
        assert float(r["losses"][r["best"]]) <= 1e-10
        np.testing.assert_allclose(r["plan"][:, 0], np.asarray(c["expected"])[:, 0], atol=1e-5)
    B = 128
    batch = synthetic.make_batch(B, seed=5)
    w = batch["weights"][batch["weight_idx"]]
    start = O.generate_plan_batch(O.OracleParams(n_iter=0), batch["world"], w)        # loss of the raw starts
    sgd = O.generate_plan_batch(O.OracleParams(), batch["world"], w)
    lb = O.generate_plan_batch(O.OracleParams(optimizer=1, n_iter=40), batch["world"], w)
    assert np.all(lb["losses"] <= start["losses"] + 1e-6 * np.maximum(1.0, np.abs(start["losses"])))
    assert np.mean(lb["losses"].min(1) <= sgd["losses"].min(1) + 1e-5) >= 0.8


def test_generate_plan_golden_scenarios():
    for c in load_golden("plans.json")["cases"]:
        spec = O.scenario_params(c["scenario"])
        oc = None
        if spec.params.other_mode == 1:
            sc = spec.scenario
            oc = [[(sc.plan[j][t] if t < len(sc.plan[j]) else sc.control[j]) for t in range(spec.params.H)]
                  for j in range(spec.params.C - 1)]
        r = O.generate_plan(spec.params, c["world_state"], c["weights_normalised"], other_controls=oc)
        np.testing.assert_allclose(r["plan"], np.asarray(c["plan"], F32), atol=5e-6)
        np.testing.assert_allclose(r["plan"][0], np.asarray(c["control"], F32), atol=5e-6)


EPISODES = ["episode_finite_horizon_true_full.json", "episode_finite_horizon_tuned_full.json",
            "episode_finite_horizon_true_extra_inits.json", "episode_finite_horizon_true_h6.json",
            "episode_local_opt_true_full.json", "episode_local_opt_tuned_full.json",
            "episode_local_opt_scaled_short.json", "episode_local_opt_true_extra_inits.json",
            "episode_replanning_true_full.json", "episode_replanning_tuned_full.json"]


@pytest.mark.parametrize("fname", EPISODES)
def test_episode_golden(fname):
    e = load_golden(fname)
    spec = O.scenario_params(e["scenario"], horizon=e["horizon"], extra_inits=e["extra_inits"])
    assert spec.params.n_iter == e["n_iter"]
    for smp in e["samples"]:
        r = O.episode(spec.params, spec.scenario, np.asarray(e["init"], F32), e["plan_weights"], e["true_weights"],
                      e["T"], unlucky_idx=smp["unlucky_car_idx"])
        assert abs(r["ret"] - smp["return"]) <= 2e-6 * abs(smp["return"])
        np.testing.assert_allclose(r["controls"], np.asarray(smp["controls"], F32), atol=5e-6)
        np.testing.assert_allclose(r["states"][:, 0], np.asarray(smp["robot_states"], F32), atol=5e-6)
        for j, os_ in enumerate(smp["other_states"]):
            np.testing.assert_allclose(r["states"][:, j + 1], np.asarray(os_, F32), atol=2e-6)


def test_survey_cross_check_returns():
    """SURVEY.md Appendix D: a second, independent reading of the reference gave these returns."""
    want = {"finite_horizon": [-0.04167331475764513], "local_opt": [-0.6909196190536022],
            "replanning": [-1.0614905506372452, -0.16572473291307688]}
    for name, rets in want.items():
        spec = O.scenario_params(name)
        w = spec.designer_weights / np.linalg.norm(spec.designer_weights)
        for k, ret in enumerate(rets):
            r = O.episode(spec.params, spec.scenario, spec.example_init, w, w, spec.eval_horizon, unlucky_idx=k + 1)
            assert abs(r["ret"] - ret) <= 5e-6 * abs(ret)


def test_batch_entry_points_match_scalar_ones():
    spec = O.scenario_params("replanning")
    w = (spec.designer_weights / np.linalg.norm(spec.designer_weights)).astype(F32)
    ri = np.tile(spec.example_init, (6, 1)).astype(F32)
    ri[:, 0] += np.linspace(-0.003, 0.003, 6, dtype=F32)
    ul = np.array([1, 2, 1, 2, 1, 2], np.int32)
    batch = O.episode_batch(spec.params, spec.scenario, ri, w, w, 8, unlucky_idx=ul)
    for b in range(6):
        one = O.episode(spec.params, spec.scenario, ri[b], w, w, 8, unlucky_idx=int(ul[b]))
        assert batch[b] == one["ret"]


@pytest.mark.parametrize("part", ["primitives", "features", "planner_kats"])
def test_golden_files_regenerate_from_the_reference(part, tmp_path):
    """Where a checkout of the reference (avikj/L4DC-MPC-OCD) is named by L4DC_REFERENCE_DIR, re-run the
    generator -- the reference's unmodified Python on oracle/tf_shim -- and require the committed fixtures
    bit for bit.  The reference is not part of this repository; without it the fixtures stay as committed."""
    import json
    import os
    import subprocess
    import sys
    from pathlib import Path
    ref = os.environ.get("L4DC_REFERENCE_DIR", "")
    if not ref or not os.path.isdir(os.path.join(ref, "interact_drive")):
        pytest.skip("L4DC_REFERENCE_DIR does not name a checkout of the reference")
    root = Path(__file__).resolve().parent.parent
    subprocess.run([sys.executable, str(root / "tests" / "golden" / "make_golden.py"), "--part", part,
                    "--reference", ref, "--outdir", str(tmp_path)], check=True, capture_output=True, timeout=600)
    new = json.load(open(tmp_path / f"{part}.json"))
    old = load_golden(f"{part}.json")
    for d in (new, old):
        d.pop("generator_seconds", None)
    assert new == old


# ---- the opt-in L-BFGS: ring-buffer semantics (a rejected pair must not overwrite a live one) -----------------------
M, LS = 4, 6
def lbfgs_py(op, world, w, u0, buggy=False, log=None):
    """float64 restatement of the engine's L-BFGS for ONE start (oracle/ocd_oracle_impl.inc ocdo_lbfgs_start)."""
    n = 2 * op.H
    def fg(u, grad=True):
        r = O.mpc_reward(op, world, u.reshape(op.H, 2), w, dtype=np.float64, grad=grad)
        return (-r[0], -r[1].reshape(-1)) if grad else -r
    u = u0.copy(); f, g = fg(u)
    S = np.zeros((M, n)); Y = np.zeros((M, n)); rho = np.zeros(M)
    k = head = 0; sy_last, yy_last = 0.0, 1.0
    for it in range(op.n_iter):
        q = g.copy(); al = np.zeros(M)
        for i in range(k):
            idx = (head - 1 - i + 2 * M) % M
            dot = 0.0
            for j in range(n): dot += S[idx][j] * q[j]
            al[i] = rho[idx] * dot
            q -= al[i] * Y[idx]
        gamma = sy_last / yy_last if k > 0 else op.lr
        q = gamma * q
        for i in range(k - 1, -1, -1):
            idx = (head - 1 - i + 2 * M) % M
            dot = 0.0
            for j in range(n): dot += Y[idx][j] * q[j]
            b = rho[idx] * dot
            q += S[idx] * (al[i] - b)
        d = -q; gd = 0.0
        for j in range(n): gd += g[j] * d[j]
        if not (gd < 0):
            k = 0; d = -op.lr * g; gd = 0.0
            for j in range(n): gd += g[j] * d[j]
        if not (gd < 0): break
        t = 1.0; ok = False
        for ls in range(LS):
            ut = u + t * d
            ft = fg(ut, False)
            if ft <= f + (1e-4 * t) * gd: ok = True; break
            t *= 0.5
        if not ok: break
        ft2, gt = fg(ut)
        sj = ut - u; yj = gt - g
        if buggy:
            S[head] = sj; Y[head] = yj
        sy = 0.0; yy = 0.0
        for j in range(n): sy += sj[j] * yj[j]; yy += yj[j] * yj[j]
        if yy > 0 and sy > 1e-10 * yy:
            S[head] = sj; Y[head] = yj
            rho[head] = 1.0 / sy; head = (head + 1) % M
            if k < M: k += 1
            sy_last, yy_last = sy, yy
        elif log is not None:
            log.append((it, k))
        u, g, f = ut, gt, ft
    return u



def test_lbfgs_rejected_pair_keeps_the_live_pairs():
    """With an Armijo-only line search on a non-convex objective the curvature test s.y > 1e-10 y.y fails now and then.
    Once the ring of 4 pairs is full, slot `head` holds the OLDEST LIVE pair; a rejected candidate must leave it alone
    (round 1 wrote the candidate there first: later directions were built on a corrupted pair).  A statement-for-
    statement Python restatement of the algorithm locates starts where a rejection follows a full ring, and the C twin
    of the kernel must take exactly the fixed path there -- which differs grossly from the overwriting one."""
    op = O.OracleParams(H=5, C=2, n_iter=30, optimizer=1)
    b = synthetic.make_batch(400, seed=3)
    starts = ((0.0, 0.0), (0.0, -0.65), (0.0, 0.65))
    hit = 0
    for i, s in ((1, 2), (7, 2), (8, 1)):
        w = b["weights"][b["weight_idx"][i]].astype(np.float64)
        world = b["world"][i].astype(np.float64)
        u0 = np.tile(starts[s], op.H).astype(np.float64)
        log = []
        fixed = lbfgs_py(op, world, w, u0, log=log)
        assert any(k == M for _, k in log), "expected a rejected pair after the ring filled up"
        wrong = lbfgs_py(op, world, w, u0, buggy=True)
        got = O.generate_plan(op, world, w, dtype=np.float64, all_plans=True)["all_plans"][s].reshape(-1)
        np.testing.assert_allclose(got, fixed, rtol=0, atol=1e-9)
        hit += int(np.abs(fixed - wrong).max() > 1e-3)
    assert hit == 3
