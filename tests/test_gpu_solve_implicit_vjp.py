"""ocd_solve_implicit_vjp_batch, Engine.solve_implicit_vjp_soa and the L-BFGS branch of torch.ops.ocd_b200.solve's
autograd formula on the GPU.

Two independent routes, both through the f64 CPU oracle:
- the implicit-function formula itself at the GPU's own plan: the reduced Hessian and the mixed derivatives of the
  oracle's f64 reward gradient by central differences, and a numpy solve -- this checks the kernel whatever L-BFGS's
  convergence;
- the whole chain: central differences of the oracle's f64 L-BFGS plan (the start the GPU picked) on problems where
  that run is converged and reproducible."""
import ctypes as C

import numpy as np
import pytest
import torch

import oracle as O

pytestmark = pytest.mark.gpu

import l4dc_mpc_ocd_b200 as ocd            # noqa: E402
from l4dc_mpc_ocd_b200 import synthetic    # noqa: E402
from l4dc_mpc_ocd_b200 import torch_ops as T    # noqa: E402

from test_gpu_parity import _pp    # noqa: E402

N = ocd._native

# test_lbfgs_vs_oracle's shapes: (H, C, lanes, other_mode, extra)
SHAPES = [(5, 2, 3, 0, False), (5, 3, 2, 1, False), (6, 2, 3, 0, True), (3, 4, 3, 0, False), (16, 2, 3, 0, False)]
COND_MAX = 1e5          # reduced Hessians above this condition number are not compared (f32 entries, f64 solve)


def _problem(H, C, lanes, other_mode, extra, n_iter, B, seed):
    lane_x = (-0.1, 0.0, 0.1) if lanes == 3 else (-0.05, 0.05)
    batch = synthetic.make_batch(B, C=C, lane_x=lane_x, seed=seed)
    oc = 0.3 * synthetic.make_other_controls(B, C, H) if other_mode else None
    op = O.OracleParams(H=H, C=C, lane_x=lane_x, n_iter=n_iter, num_lanes=lanes, other_mode=other_mode,
                        extra_inits=extra, target_speed=1.0 if lanes == 3 else 1.2, lr=0.1, optimizer=1)
    p = _pp(op, ocd.MATH_PRECISE)
    p.optimizer = ocd.OPT_LBFGS
    return op, p, batch, oc


def _soa(engine, batch, oc):
    dev = engine.device
    world = torch.as_tensor(batch["world"], device=dev).permute(1, 2, 0).contiguous()
    w = torch.as_tensor(batch["weights"], device=dev).t().contiguous()
    idx = torch.as_tensor(batch["weight_idx"], device=dev)
    ocs = None if oc is None else torch.as_tensor(oc, device=dev).permute(1, 2, 3, 0).contiguous()
    return world, w, idx, ocs


def _solve_and_ivjp(engine, p, batch, oc, plan_bar, residual=True):
    """-> (forward result in SoA, plan [B, H, 2], weights_bar [B, K], world_bar [B, C, 4], residual [B])."""
    world, w, idx, ocs = _soa(engine, batch, oc)
    B = world.shape[-1]
    Bo = 0 if ocs is None else B
    fwd = engine.solve_soa(p, world, w, w.shape[1], idx, ocs, Bo)
    pb = torch.as_tensor(plan_bar, device=engine.device).permute(1, 2, 0).contiguous()
    out = engine.solve_implicit_vjp_soa(p, world, w, w.shape[1], fwd["plan"], pb, idx, ocs, Bo, residual=residual)
    plan = fwd["plan"].permute(2, 0, 1).cpu().numpy()
    wb = out["weights_bar"].t().cpu().numpy().astype(np.float64)
    xb = out["world_bar"].permute(2, 0, 1).cpu().numpy().astype(np.float64)
    res = out["residual"].cpu().numpy() if residual else None
    return fwd, plan, wb, xb, res


def _active(u):
    """Flat indices (2t + c) of the controls inside the inclusive clip box."""
    u = np.asarray(u).reshape(-1)
    a, om = u[0::2], u[1::2]
    m = np.zeros(u.size, bool)
    m[0::2] = (a >= -8.0) & (a <= 4.0)
    m[1::2] = np.abs(om) <= 4.0
    return np.nonzero(m)[0]


def _grad64(op, x, u, w, oc):
    _, g = O.mpc_reward(op, x, u.reshape(op.H, 2), w, other_controls=oc, dtype=np.float64)
    return np.asarray(g, np.float64).reshape(-1)


def _ift_reference(op, x, u, w, oc, act, pbar, dw, dx, h):
    """Host f64 IFT at the plan u: -> (<theta_bar, (dw, dx)>, cond(H_AA)) with H_AA and dG_A/dtheta along (dw, dx) by
    central differences (step h) of the oracle's reward gradient."""
    n = len(act)
    Hm = np.zeros((n, n))
    for j, c in enumerate(act):
        e = np.zeros(u.size)
        e[c] = h
        Hm[:, j] = (_grad64(op, x, u + e, w, oc) - _grad64(op, x, u - e, w, oc))[act] / (2 * h)
    Hm = 0.5 * (Hm + Hm.T)
    cond = float(np.linalg.cond(Hm))
    if not cond <= COND_MAX:
        return np.nan, cond
    Gt = (_grad64(op, x + h * dx, u, w + h * dw, oc) - _grad64(op, x - h * dx, u, w - h * dw, oc))[act] / (2 * h)
    z = np.linalg.solve(Hm, pbar[act])
    return -float(z @ Gt), cond


@pytest.mark.parametrize("H,C,lanes,other_mode,extra", SHAPES)
def test_ift_formula_at_the_gpus_plan(engine, H, C, lanes, other_mode, extra):
    """weights_bar and world_bar in random directions against the IFT assembled on the host from the oracle's f64
    reward gradient at the GPU's plan.  Skipped: a problem whose two step sizes disagree (a kink of the gradient,
    e.g. a min / max switch, within the step) or whose reduced Hessian has a condition number above COND_MAX.  On
    these random batches many reduced Hessians are exactly singular (an active control the reward does not depend on,
    such as the last steering with the speed feature saturated); the kernel must return NaN exactly on problems the
    host finds singular or ill-conditioned."""
    B = 128
    op, p, batch, oc = _problem(H, C, lanes, other_mode, extra, 40, B, seed=17 * H + C)
    rng = np.random.default_rng(H + 10 * C)
    pbar = rng.normal(size=(B, H, 2)).astype(np.float32)
    _, plan, wb, xb, _ = _solve_and_ivjp(engine, p, batch, oc, pbar)
    w_full = batch["weights"][batch["weight_idx"]].astype(np.float64)
    errs, kinks, illc = [], 0, 0
    for b in range(B):
        u = plan[b].astype(np.float64).reshape(-1)
        act = _active(u)
        if len(act) == 0:
            continue
        x = batch["world"][b].astype(np.float64)
        ocb = None if oc is None else oc[b].astype(np.float64)
        dw = rng.normal(size=p.K)
        dx = rng.normal(size=(C, 4)) * np.array([0.02, 0.02, 0.1, 0.05])
        pb = pbar[b].astype(np.float64).reshape(-1)
        q1, cond = _ift_reference(op, x, u, w_full[b], ocb, act, pb, dw, dx, 1e-5)
        if np.isnan(wb[b]).any():
            assert not cond <= COND_MAX, (b, cond)           # singular on the GPU: singular or ill-conditioned here
            illc += 1
            continue
        if not cond <= COND_MAX:
            illc += 1
            continue
        q2, _ = _ift_reference(op, x, u, w_full[b], ocb, act, pb, dw, dx, 5e-6)
        scale = max(abs(q2), 1e-2)
        if abs(q1 - q2) > 1e-3 * scale:
            kinks += 1
            continue
        got = float(wb[b] @ dw + np.sum(xb[b] * dx))
        errs.append(abs(got - q2) / scale)
    errs = np.asarray(errs)
    print(f"H={H} C={C}: {len(errs)} checked, {kinks} at a kink, {illc} ill-conditioned, "
          f"median {np.median(errs):.2e}, worst {errs.max():.2e}")
    assert len(errs) >= 8 and kinks <= 0.25 * (len(errs) + kinks), (len(errs), kinks, illc)
    assert np.median(errs) <= 1e-3
    assert np.mean(errs <= 2e-2) >= 0.95, np.sort(errs)[-5:]


@pytest.mark.parametrize("H,C,lanes,other_mode,extra", SHAPES)
def test_vjp_vs_oracle_lbfgs_differences(engine, H, C, lanes, other_mode, extra):
    """End to end: the derivative of the oracle's f64 L-BFGS plan (the start the GPU picked, n_iter 400) by central
    differences in random directions, on problems where that f64 run is converged (max |G_A| < 1e-6), reproducible
    under the parity test's ulp probe, and where the GPU found the same optimum: the same active set and its controls
    within 1e-3.  plan_bar lives on the active set: a clipped control's value beyond the box is arbitrary (it keeps
    whatever the L-BFGS history moved it by), and its derivative is zero by construction.  At H = 16 the f32 run
    rarely reaches the f64 optimum in 100 iterations, so only a few problems qualify there."""
    B = 96 if H < 16 else 256
    op, p, batch, oc = _problem(H, C, lanes, other_mode, extra, 100, B, seed=29 * H + C)
    op64 = O.OracleParams(**{**op.__dict__, "n_iter": 400})
    rng = np.random.default_rng(3 * H + C)
    world, w, idx, ocs = _soa(engine, batch, oc)
    Bo = 0 if ocs is None else B
    fwd = engine.solve_soa(p, world, w, w.shape[1], idx, ocs, Bo)
    plan = fwd["plan"].permute(2, 0, 1).cpu().numpy()
    pbar = rng.normal(size=(B, H, 2)).astype(np.float32)
    for b in range(B):
        m = np.zeros(2 * H, np.float32)
        m[_active(plan[b])] = 1.0
        pbar[b] *= m.reshape(H, 2)
    out = engine.solve_implicit_vjp_soa(p, world, w, w.shape[1], fwd["plan"],
                                        torch.as_tensor(pbar, device=engine.device).permute(1, 2, 0).contiguous(), idx,
                                        ocs, Bo)
    wb = out["weights_bar"].t().cpu().numpy().astype(np.float64)
    xb = out["world_bar"].permute(2, 0, 1).cpu().numpy().astype(np.float64)
    best = fwd["best"].cpu().numpy()
    w_full = batch["weights"][batch["weight_idx"]].astype(np.float64)

    def plan64(b, x, w):
        ocb = None if oc is None else oc[b].astype(np.float64)
        r = O.generate_plan(op64, x, w, other_controls=ocb, dtype=np.float64, all_plans=True)
        return np.asarray(r["all_plans"])[best[b]].reshape(-1)
    errs, kinks, candidates = [], 0, 0
    for b in range(B):
        x = batch["world"][b].astype(np.float64)
        u64 = plan64(b, x, w_full[b])
        act = _active(u64)
        ocb = None if oc is None else oc[b].astype(np.float64)
        if len(act) == 0 or np.abs(_grad64(op64, x, u64, w_full[b], ocb)[act]).max() >= 1e-6:
            continue
        if not np.array_equal(_active(plan[b]), act) or np.abs(plan[b].reshape(-1) - u64)[act].max() >= 1e-3:
            continue
        if np.isnan(wb[b]).any():
            continue
        reproducible = True
        for col, eps in ((0, 3e-8), (3, -2.4e-7), (2, 1.2e-7)):
            xp = x.copy()
            xp[0, col] += eps
            if np.abs(plan64(b, xp, w_full[b]) - u64)[act].max() > 1e-5:
                reproducible = False
                break
        if not reproducible:
            continue
        candidates += 1
        dw = rng.normal(size=p.K)
        dx = rng.normal(size=(C, 4)) * np.array([0.02, 0.02, 0.1, 0.05])
        pb = pbar[b].astype(np.float64).reshape(-1)

        def q(h):
            return float(pb @ (plan64(b, x + h * dx, w_full[b] + h * dw) - plan64(b, x - h * dx, w_full[b] - h * dw))
                         / (2 * h))
        q1, q2 = q(1e-5), q(5e-6)
        scale = max(abs(q2), 1e-2)
        if abs(q1 - q2) > 1e-3 * scale:
            kinks += 1
            continue
        got = float(wb[b] @ dw + np.sum(xb[b] * dx))
        errs.append(abs(got - q2) / scale)
    errs = np.asarray(errs)
    print(f"H={H} C={C}: {candidates} converged and reproducible, {len(errs)} checked, {kinks} at a kink, "
          f"median {np.median(errs) if len(errs) else np.nan:.2e}, worst {errs.max() if len(errs) else np.nan:.2e}")
    if H == 16 and candidates == 0:
        pytest.skip("no problem where the f32 L-BFGS run reached the converged f64 optimum (the IFT formula itself is "
                    "checked at H = 16 by test_ift_formula_at_the_gpus_plan)")
    assert len(errs) >= (8 if H < 16 else 1) and len(errs) >= 0.6 * candidates, (len(errs), candidates, kinks)
    assert np.median(errs) <= 1e-3
    assert np.mean(errs <= 2e-2) >= 0.95, np.sort(errs)[-5:]


@pytest.mark.parametrize("n_iter", [2, 100])
@pytest.mark.parametrize("H,C,lanes,other_mode,extra", SHAPES)
def test_residual_is_the_masked_reward_gradient(engine, n_iter, H, C, lanes, other_mode, extra):
    """residual = max over the unclipped controls of |d reward / d controls| at the plan (Engine.reward's gradient),
    both far from stationarity (2 iterations) and near it (100)."""
    B = 256
    op, p, batch, oc = _problem(H, C, lanes, other_mode, extra, n_iter, B, seed=5 * H + C)
    _, plan, _, _, res = _solve_and_ivjp(engine, p, batch, oc, np.ones((B, H, 2), np.float32))
    _, G = engine.reward(p, batch["world"], plan, batch["weights"], weight_idx=batch["weight_idx"], other_controls=oc)
    G = G.cpu().numpy().reshape(B, -1)
    want = np.zeros(B)
    for b in range(B):
        act = _active(plan[b])
        want[b] = np.abs(G[b, act]).max() if len(act) else 0.0
    gscale = np.abs(G).max(1)
    assert np.all(np.abs(res - want) <= 1e-4 * want + 1e-6 * np.maximum(1.0, gscale)), \
        np.sort(np.abs(res - want))[-5:]


def test_clipped_controls_have_zero_derivative(engine):
    """Plans that saturate the acceleration at every step (the extra-init starts from a speed whose friction term
    exceeds the box: L-BFGS never moves a clipped control): a plan_bar on the clipped coordinates alone gives exactly
    zero, one on the active coordinates does not."""
    H, Cc = 5, 2
    op, p, batch, _ = _problem(H, Cc, 3, 0, True, 40, 64, seed=4)
    world, w, idx, _ = _soa(engine, batch, None)
    B = world.shape[-1]
    cs = torch.full((B,), 6.0, device=engine.device)          # a0 = 0.2 * 36 = 7.2 > 4
    fwd = engine.solve_soa(p, world, w, w.shape[1], idx, cur_speed=cs, all_plans=True)
    plan = fwd["all_plans"][3].contiguous()                   # start 3: a0, no turn
    assert (plan[:, 0, :] > 4.0).all()
    on_acc = torch.zeros((H, 2, B), device=engine.device)
    on_acc[:, 0, :] = torch.as_tensor(np.random.default_rng(0).normal(size=(H, B)), dtype=torch.float32)
    out = engine.solve_implicit_vjp_soa(p, world, w, w.shape[1], plan, on_acc, idx)
    assert (out["weights_bar"] == 0).all() and (out["world_bar"] == 0).all()
    on_ang = torch.zeros((H, 2, B), device=engine.device)
    on_ang[:, 1, :] = 1.0
    out = engine.solve_implicit_vjp_soa(p, world, w, w.shape[1], plan, on_ang, idx)
    fin = torch.isfinite(out["weights_bar"]).all(0)
    assert fin.float().mean() >= 0.5 and (out["weights_bar"][:, fin].abs().sum(0) > 0).float().mean() >= 0.5


def test_singular_problem_is_nan_and_isolated(engine):
    """A problem with all-zero weights has a zero reduced Hessian: its rows are NaN, and every other problem's rows
    are bit for bit those of a batch without it."""
    H, Cc, B = 5, 2, 48
    op, p, batch, _ = _problem(H, Cc, 3, 0, False, 40, B, seed=9)
    world, w, idx, _ = _soa(engine, batch, None)
    wfull = w[:, idx.long()].contiguous()                     # one vector per problem
    fwd = engine.solve_soa(p, world, wfull, B)
    pb = torch.as_tensor(np.random.default_rng(2).normal(size=(H, 2, B)), dtype=torch.float32, device=engine.device)
    ref = engine.solve_implicit_vjp_soa(p, world, wfull, B, fwd["plan"], pb, residual=True)
    j = 17
    wz = wfull.clone()
    wz[:, j] = 0.0
    plan = fwd["plan"].clone()
    plan[:, :, j] = engine.solve_soa(p, world, wz, B)["plan"][:, :, j]
    out = engine.solve_implicit_vjp_soa(p, world, wz, B, plan, pb, residual=True)
    assert torch.isnan(out["weights_bar"][:, j]).all() and torch.isnan(out["world_bar"][:, :, j]).all()
    assert out["residual"][j] == 0
    keep = torch.arange(B, device=engine.device) != j
    for k in ("weights_bar", "world_bar", "residual"):        # bit for bit, NaN rows of other problems included
        assert torch.equal(out[k][..., keep].view(torch.int32), ref[k][..., keep].view(torch.int32)), k


@pytest.mark.parametrize("B", [1, 127, 129, 1000])
@pytest.mark.parametrize("with_world_bar,with_residual", [(True, True), (False, False), (True, False), (False, True)])
def test_outputs_stay_in_bounds(engine, B, with_world_bar, with_residual):
    """Every output sits inside a sentinel-filled buffer at ragged batch sizes: the guard bands survive and each
    window is fully written; outputs passed as NULL are not written."""
    H, Cc = 6, 3
    batch = synthetic.make_batch(B, C=Cc, seed=B)
    p = ocd.PlannerParams(H=H, C=Cc, n_iter=20, extra_inits=True, optimizer=ocd.OPT_LBFGS)
    world, w, idx, _ = _soa(engine, batch, None)
    fwd = engine.solve_soa(p, world, w, w.shape[1], idx)
    pb = torch.as_tensor(np.random.default_rng(B).normal(size=(H, 2, B)), dtype=torch.float32, device=engine.device)
    G, SENT = 1024, 12345.0
    sizes = dict(wbar=p.K * B, xbar=p.C * 4 * B, res=B)
    bufs = {k: torch.full((n + 2 * G,), SENT, dtype=torch.float32, device=engine.device) for k, n in sizes.items()}
    win = {k: bufs[k][G:G + n] for k, n in sizes.items()}
    ptr = lambda t: C.c_void_p(t.data_ptr())
    ps = p.c_struct()
    rc = N.lib.ocd_solve_implicit_vjp_batch(C.addressof(ps), ptr(world), None, 0, ptr(w), w.shape[1], ptr(idx),
                                            ptr(fwd["plan"]), ptr(pb), ptr(win["wbar"]),
                                            ptr(win["xbar"]) if with_world_bar else None,
                                            ptr(win["res"]) if with_residual else None, B,
                                            C.c_void_p(torch.cuda.current_stream().cuda_stream))
    N.check(rc, "ocd_solve_implicit_vjp_batch")
    torch.cuda.synchronize()
    written = dict(wbar=True, xbar=with_world_bar, res=with_residual)
    for k, buf in bufs.items():
        n = win[k].numel()
        assert (buf[:G] == SENT).all() and (buf[G + n:] == SENT).all(), k
        if written[k]:
            assert (buf[G:G + n] != SENT).all(), k
        else:
            assert (buf[G:G + n] == SENT).all(), k


# ---- autograd -----------------------------------------------------------------------------------------------------
def test_autograd_matches_the_engine(engine):
    p = ocd.PlannerParams(extra_inits=True, n_iter=40, optimizer=ocd.OPT_LBFGS)
    batch = synthetic.make_batch(120, seed=8)           # Bw = B / 5 vectors, weight_idx
    world, w, idx, _ = _soa(engine, batch, None)
    B, Bw = world.shape[-1], w.shape[1]
    assert Bw < B
    wg, xg = w.clone().requires_grad_(True), world.clone().requires_grad_(True)
    plan, losses, best = torch.ops.ocd_b200.solve(xg, wg, idx, None, T.pack_params(p))
    pb = torch.as_tensor(np.random.default_rng(1).normal(size=tuple(plan.shape)), dtype=torch.float32,
                         device=engine.device)
    gw, gx = torch.autograd.grad(plan, (wg, xg), pb, retain_graph=True)
    gw2, gx2 = torch.autograd.grad(plan, (wg, xg), pb)
    bits = lambda t: t.contiguous().view(torch.int32)              # singular problems' rows are NaN
    assert torch.equal(bits(gw), bits(gw2)) and torch.equal(bits(gx), bits(gx2))   # deterministic, bit for bit
    ref = engine.solve_implicit_vjp_soa(p, world, w, Bw, plan.detach().contiguous(), pb, idx)
    assert torch.equal(bits(gx), bits(ref["world_bar"]))
    per = ref["weights_bar"].cpu().numpy().astype(np.float64)     # [K][B], per problem
    want = np.zeros((p.K, Bw))
    for b in range(B):
        want[:, batch["weight_idx"][b]] += per[:, b]
    got = gw.cpu().numpy()
    fin = np.isfinite(want).all(0)
    assert np.array_equal(np.isfinite(got).all(0), fin)
    np.testing.assert_allclose(got[:, fin], want[:, fin], rtol=1e-5, atol=1e-5 * np.abs(want[:, fin]).max())


def test_autograd_refuses_what_it_cannot_differentiate(engine):
    p = ocd.PlannerParams(n_iter=20, optimizer=ocd.OPT_LBFGS)
    batch = synthetic.make_batch(40, seed=8)
    world, w, idx, _ = _soa(engine, batch, None)
    wg = w.clone().requires_grad_(True)
    plan, losses, _ = torch.ops.ocd_b200.solve(world, wg, idx, None, T.pack_params(p))
    with pytest.raises(RuntimeError, match="losses"):
        (plan.sum() + losses.sum()).backward()
    spec = O.scenario_params("replanning")
    pr = _pp(spec.params, ocd.MATH_PRECISE)
    pr.optimizer = ocd.OPT_LBFGS
    B = 8
    wr = torch.as_tensor(np.tile(spec.designer_weights / np.linalg.norm(spec.designer_weights), (B, 1)).T.copy(),
                         dtype=torch.float32, device=engine.device).requires_grad_(True)
    wo = torch.as_tensor(np.tile(np.concatenate([[spec.example_init], spec.scenario.init_state]), (B, 1, 1)),
                         dtype=torch.float32, device=engine.device).permute(1, 2, 0).contiguous()
    oc = torch.zeros((pr.C - 1, pr.H, 2, B), device=engine.device, requires_grad=True)
    plan, _, _ = torch.ops.ocd_b200.solve(wo, wr, None, oc, T.pack_params(pr))
    with pytest.raises(RuntimeError, match="other_controls"):
        plan.sum().backward()

