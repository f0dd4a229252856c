"""ocd_solve_vjp_batch, Engine.solve_vjp_soa and the autograd formula of torch.ops.ocd_b200.solve on the GPU.

The independent route is the f64 CPU oracle: the plan of the start the GPU picked, differenced in random directions of
the weights and of the whole initial world.  Full-budget runs are checked on the problems the parity tests' probe
(solve_conditioning) finds reproducible; at two iterations every problem is checked."""
import ctypes as C

import numpy as np
import pytest
import torch

import oracle as O

pytestmark = pytest.mark.gpu

import l4dc_mpc_ocd_b200 as ocd            # noqa: E402
from l4dc_mpc_ocd_b200 import synthetic    # noqa: E402
from l4dc_mpc_ocd_b200 import torch_ops as T    # noqa: E402

from test_gpu_parity import MODES, _pp, solve_conditioning    # noqa: E402

N = ocd._native


def _problem(H, C, lanes, other_mode, extra, n_iter, lr, B, seed):
    lane_x = (-0.1, 0.0, 0.1) if lanes == 3 else (-0.05, 0.05)
    batch = synthetic.make_batch(B, C=C, lane_x=lane_x, seed=seed)
    oc = 0.3 * synthetic.make_other_controls(B, C, H) if other_mode else None
    op = O.OracleParams(H=H, C=C, lane_x=lane_x, n_iter=n_iter, num_lanes=lanes, other_mode=other_mode,
                        extra_inits=extra, target_speed=1.0 if lanes == 3 else 1.2, lr=lr)
    return op, batch, oc


def _soa(engine, batch, oc):
    dev = engine.device
    world = torch.as_tensor(batch["world"], device=dev).permute(1, 2, 0).contiguous()
    w = torch.as_tensor(batch["weights"], device=dev).t().contiguous()
    idx = torch.as_tensor(batch["weight_idx"], device=dev)
    ocs = None if oc is None else torch.as_tensor(oc, device=dev).permute(1, 2, 3, 0).contiguous()
    return world, w, idx, ocs


def _solve_and_vjp(engine, p, batch, oc, plan_bar, world_bar=True):
    """-> (forward result in SoA, weights_bar [B, K] per problem, world_bar [B, C, 4])."""
    world, w, idx, ocs = _soa(engine, batch, oc)
    B = world.shape[-1]
    Bo = 0 if ocs is None else B
    fwd = engine.solve_soa(p, world, w, w.shape[1], idx, ocs, Bo)
    pb = torch.as_tensor(plan_bar, device=engine.device).permute(1, 2, 0).contiguous()
    out = engine.solve_vjp_soa(p, world, w, w.shape[1], fwd["best"], pb, idx, ocs, Bo, world_bar=world_bar)
    wb = out["weights_bar"].t().cpu().numpy().astype(np.float64)
    xb = out["world_bar"].permute(2, 0, 1).cpu().numpy().astype(np.float64) if world_bar else None
    return fwd, wb, xb


def _directional(op, batch, oc, b, best, dw, dx, pbar, h):
    """<plan_bar, central difference of the f64 oracle's plan of start `best`> along (dw, dx), step h."""
    w64 = batch["weights"][batch["weight_idx"][b]].astype(np.float64)
    x64 = batch["world"][b].astype(np.float64)
    ocb = None if oc is None else oc[b].astype(np.float64)

    def plan(sgn):
        r = O.generate_plan(op, x64 + sgn * h * dx, w64 + sgn * h * dw, other_controls=ocb, dtype=np.float64,
                            all_plans=True)
        return np.asarray(r["all_plans"])[best]
    return float(np.sum(pbar * (plan(1.0) - plan(-1.0)) / (2 * h)))


def _compare(op, batch, oc, probs, best, wb, xb, rng, h):
    """For each problem: random directions over every weight and every component of every car; -> (rel errors of the
    checked problems, number skipped at a kink)."""
    errs, skipped = [], 0
    for b in probs:
        dw = rng.normal(size=wb.shape[1])
        dx = rng.normal(size=xb.shape[1:]) * np.array([0.02, 0.02, 0.1, 0.05])
        pbar = _compare.pbar[b]
        q1 = _directional(op, batch, oc, b, int(best[b]), dw, dx, pbar, h)
        q2 = _directional(op, batch, oc, b, int(best[b]), dw, dx, pbar, h / 2)
        scale = max(abs(q1), 1e-2)
        if abs(q1 - q2) > 1e-3 * scale:         # a kink inside the interval: the quotient means nothing there
            skipped += 1
            continue
        got = float(np.dot(wb[b], dw) + np.sum(xb[b] * dx))
        errs.append(abs(got - q2) / scale)
    return np.asarray(errs), skipped


SHAPES = [(5, 2, 3, 0, False, 100, 0.1),     # finite_horizon
          (5, 3, 2, 1, False, 100, 0.1),     # replanning
          (6, 2, 3, 0, True, 200, 0.1),      # extra-init starts: the start depends on v0
          (15, 2, 3, 0, False, 100, 0.02),   # medium horizon
          (8, 5, 3, 0, False, 100, 0.1)]     # four other cars


@pytest.mark.parametrize("mode,_n", MODES)
@pytest.mark.parametrize("H,C,lanes,other_mode,extra,n_iter,lr", SHAPES)
def test_vjp_vs_oracle_differences(engine, mode, _n, H, C, lanes, other_mode, extra, n_iter, lr):
    B = 96
    op, batch, oc = _problem(H, C, lanes, other_mode, extra, n_iter, lr, B, seed=31 * H + C)
    w_full = batch["weights"][batch["weight_idx"]]
    ref, ref64, cond_u, cond_l = solve_conditioning(op, batch["world"], w_full, oc)
    rng = np.random.default_rng(H + 10 * C)
    pbar = rng.normal(size=(B, H, 2)).astype(np.float32)
    fwd, wb, xb = _solve_and_vjp(engine, _pp(op, mode), batch, oc, pbar)
    best = fwd["best"].cpu().numpy()
    well = (cond_u < 1e-5) & (ref["best"] == ref64["best"]) & (best == ref["best"]) & (cond_l.max(1) < 1e-4)
    assert well.sum() >= 12, well.sum()
    assert np.isfinite(wb).all() and np.isfinite(xb).all()
    _compare.pbar = pbar.astype(np.float64)
    errs, skipped = _compare(op, batch, oc, np.nonzero(well)[0], best, wb, xb, rng, 1e-5)
    print(f"H={H} C={C} mode={mode}: {len(errs)} checked, {skipped} at a kink, median {np.median(errs):.2e}, "
          f"worst {errs.max():.2e}")
    assert len(errs) >= 0.8 * (len(errs) + skipped), (len(errs), skipped)
    assert np.median(errs) <= 1e-3
    assert np.mean(errs <= 2e-2) >= 0.95, np.sort(errs)[-5:]


@pytest.mark.parametrize("mode,_n", MODES)
@pytest.mark.parametrize("H,C,lanes,other_mode,extra", [(5, 2, 3, 0, False), (5, 3, 2, 1, False), (6, 2, 3, 0, True),
                                                        (8, 5, 3, 0, False), (15, 3, 3, 0, False)])
def test_two_iterations_every_problem(engine, mode, _n, H, C, lanes, other_mode, extra):
    """Two SGD iterations amplify nothing: every problem of the random batch is checked (bar a kink inside the
    differencing interval)."""
    B = 384
    op, batch, oc = _problem(H, C, lanes, other_mode, extra, 2, 0.1 if H < 15 else 0.03, B, seed=7 + H * C)
    rng = np.random.default_rng(3 * H + C)
    pbar = rng.normal(size=(B, H, 2)).astype(np.float32)
    fwd, wb, xb = _solve_and_vjp(engine, _pp(op, mode), batch, oc, pbar)
    _compare.pbar = pbar.astype(np.float64)
    errs, skipped = _compare(op, batch, oc, range(B), fwd["best"].cpu().numpy(), wb, xb, rng, 1e-6)
    assert skipped <= 0.03 * B, skipped
    assert errs.max() <= 2e-3, np.sort(errs)[-5:]


def test_full_jacobian_on_a_few_problems(engine):
    """One-hot plan_bar rows: the 2H VJPs are the rows of d plan / d w, entry by entry against difference quotients."""
    H, Cc = 5, 2
    op, batch, _ = _problem(H, Cc, 3, 0, False, 100, 0.1, 64, seed=5)
    w_full = batch["weights"][batch["weight_idx"]]
    ref, ref64, cond_u, cond_l = solve_conditioning(op, batch["world"], w_full)
    well = np.nonzero((cond_u < 1e-6) & (ref["best"] == ref64["best"]))[0][:4]
    assert len(well) == 4
    n = 2 * H
    rep = {k: np.repeat(v[well], n, axis=0) for k, v in (("world", batch["world"]),)}
    rep["weights"] = w_full[well].repeat(n, axis=0)
    rep["weight_idx"] = np.arange(4 * n, dtype=np.int32)
    pbar = np.tile(np.eye(n, dtype=np.float32).reshape(n, H, 2), (4, 1, 1))
    p = _pp(op, ocd.MATH_PRECISE)
    fwd, wb, _ = _solve_and_vjp(engine, p, rep, None, pbar, world_bar=False)
    best = fwd["best"].cpu().numpy()
    h = 1e-5
    for i, b in enumerate(well):
        jac = wb[i * n:(i + 1) * n]                          # [2H, K]: row r = d plan_r / d w
        ref_j = np.zeros_like(jac)
        for k_ in range(p.K):
            e = np.zeros(p.K); e[k_] = h
            pp = O.generate_plan(op, batch["world"][b].astype(np.float64), w_full[b] + e, dtype=np.float64, all_plans=True)
            pm = O.generate_plan(op, batch["world"][b].astype(np.float64), w_full[b] - e, dtype=np.float64, all_plans=True)
            ref_j[:, k_] = ((np.asarray(pp["all_plans"]) - np.asarray(pm["all_plans"]))[best[i * n]] / (2 * h)).reshape(n)
        np.testing.assert_allclose(jac, ref_j, atol=2e-3 * max(1.0, np.abs(ref_j).max()), rtol=0)


def test_iterates_are_the_forwards_own(engine):
    """The workspace holds u^0 .. u^{N-1} of the winning start, bit for bit those of the forward (a forward with
    n_iter = n returns u^n as all_plans), for every form of iteration code: register-resident, medium-horizon,
    segmented with compile-time and runtime horizon, in both math modes."""
    for H, Cc, lr in ((5, 2, 0.1), (15, 2, 0.02), (15, 4, 0.02), (8, 5, 0.1), (50, 2, 0.0003)):
        for mode in (ocd.MATH_FAST, ocd.MATH_PRECISE):
            if mode == ocd.MATH_PRECISE and H in (15, 50):
                continue
            B, n_iter = 97, 6
            op, batch, _ = _problem(H, Cc, 3, 0, False, n_iter, lr, B, seed=H + Cc)
            p = _pp(op, mode)
            world, w, idx, _ = _soa(engine, batch, None)
            fwd = engine.solve_soa(p, world, w, w.shape[1], idx)
            pb = torch.ones((H, 2, B), device=engine.device)
            bufs, win = _raw_vjp(engine, p, world, w, idx, fwd["best"], pb)
            its = win["ws"].view(n_iter, H, 2, B)
            best = fwd["best"].long()
            for n in (0, 1, n_iter - 1):
                q = _pp(op, mode)
                q.n_iter = n
                ap = engine.solve_soa(q, world, w, w.shape[1], idx, all_plans=True)["all_plans"]   # [S][H][2][B]
                want = ap[best, :, :, torch.arange(B, device=engine.device)]                       # [B][H][2]
                assert torch.equal(its[n].permute(2, 0, 1), want), (H, Cc, mode, n)


def _raw_vjp(engine, p, world, w, idx, best, plan_bar, G=1024, SENT=12345.0):
    """ocd_solve_vjp_batch with every output (and the workspace) a window inside a sentinel-filled buffer."""
    B = world.shape[-1]
    dev = engine.device
    ps = p.c_struct()
    nb = C.c_size_t(0)
    N.check(N.lib.ocd_solve_vjp_workspace_bytes(C.addressof(ps), B, C.byref(nb)))
    sizes = dict(wbar=p.K * B, xbar=p.C * 4 * B, ws=nb.value // 4)
    bufs = {k: torch.full((n + 2 * G,), SENT, dtype=torch.float32, device=dev) for k, n in sizes.items()}
    win = {k: bufs[k][G:G + n] for k, n in sizes.items()}
    ptr = lambda t: C.c_void_p(t.data_ptr())
    rc = N.lib.ocd_solve_vjp_batch(C.addressof(ps), ptr(world), None, 0, ptr(w), w.shape[1],
                                   None if idx is None else ptr(idx), None, ptr(best), ptr(plan_bar), ptr(win["wbar"]),
                                   ptr(win["xbar"]), ptr(win["ws"]), nb.value, B,
                                   C.c_void_p(torch.cuda.current_stream().cuda_stream))
    N.check(rc, "ocd_solve_vjp_batch")
    torch.cuda.synchronize()
    return bufs, win


@pytest.mark.parametrize("H,C,extra,B", [(5, 2, False, 33), (5, 2, True, 1), (6, 2, True, 257), (15, 2, False, 65),
                                         (15, 4, False, 130), (8, 5, False, 4097), (50, 2, False, 31),
                                         (64, 8, True, 3)])
def test_outputs_stay_in_bounds(engine, H, C, extra, B):
    """Every output and the workspace sit inside sentinel-filled buffers at ragged batch sizes: the guard bands must
    survive and each window must be fully written."""
    batch = synthetic.make_batch(B, C=C, seed=H + C)
    p = ocd.PlannerParams(H=H, C=C, n_iter=4, extra_inits=extra, lr=0.1 if H <= 8 else (0.02 if H <= 16 else 0.0003))
    world, w, idx, _ = _soa(engine, batch, None)
    fwd = engine.solve_soa(p, world, w, w.shape[1], idx)
    pb = torch.as_tensor(np.random.default_rng(B).normal(size=(H, 2, B)), dtype=torch.float32, device=engine.device)
    G, SENT = 1024, 12345.0
    bufs, win = _raw_vjp(engine, p, world, w, idx, fwd["best"], pb, G, SENT)
    for k, buf in bufs.items():
        n = win[k].numel()
        assert (buf[:G] == SENT).all() and (buf[G + n:] == SENT).all(), k
        assert (buf[G:G + n] != SENT).all(), k
    assert torch.isfinite(win["wbar"]).all() and torch.isfinite(win["xbar"]).all()


# ---- autograd -----------------------------------------------------------------------------------------------------
def _autograd_inputs(engine, B=120, seed=8):
    batch = synthetic.make_batch(B, seed=seed)           # Bw = B / 5 vectors, weight_idx
    world, w, idx, _ = _soa(engine, batch, None)
    return batch, world, w, idx


def test_autograd_matches_the_engine(engine):
    p = ocd.PlannerParams(extra_inits=True)
    batch, world, w, idx = _autograd_inputs(engine)
    B, Bw = world.shape[-1], w.shape[1]
    assert Bw < B
    with torch.no_grad():
        plain = torch.ops.ocd_b200.solve(world, w, idx, None, T.pack_params(p))
    wg, xg = w.clone().requires_grad_(True), world.clone().requires_grad_(True)
    plan, losses, best = torch.ops.ocd_b200.solve(xg, wg, idx, None, T.pack_params(p))
    for a, b_ in zip((plan, losses, best), plain):       # the forward is untouched by autograd
        assert torch.equal(a.detach(), b_)
    pb = torch.as_tensor(np.random.default_rng(1).normal(size=tuple(plan.shape)), dtype=torch.float32,
                         device=engine.device)
    gw, gx = torch.autograd.grad(plan, (wg, xg), pb, retain_graph=True)
    gw2, gx2 = torch.autograd.grad(plan, (wg, xg), pb)
    assert torch.equal(gw, gw2) and torch.equal(gx, gx2)          # deterministic, bit for bit
    ref = engine.solve_vjp_soa(p, world, w, Bw, best, pb, idx)
    assert torch.equal(gx, ref["world_bar"])
    per = ref["weights_bar"].cpu().numpy().astype(np.float64)     # [K][B], per problem
    want = np.zeros((p.K, Bw))
    for b in range(B):
        want[:, batch["weight_idx"][b]] += per[:, b]
    np.testing.assert_allclose(gw.cpu().numpy(), want, rtol=1e-5, atol=1e-5 * np.abs(want).max())


def test_autograd_refuses_what_it_cannot_differentiate(engine):
    p = ocd.PlannerParams()
    _, world, w, idx = _autograd_inputs(engine, B=40)
    wg = w.clone().requires_grad_(True)
    plan, losses, _ = torch.ops.ocd_b200.solve(world, wg, idx, None, T.pack_params(p))
    with pytest.raises(RuntimeError, match="losses"):
        (plan.sum() + losses.sum()).backward()
    spec = O.scenario_params("replanning")
    pr = _pp(spec.params, ocd.MATH_FAST)
    B = 8
    wr = torch.as_tensor(np.tile(spec.designer_weights / np.linalg.norm(spec.designer_weights), (B, 1)).T.copy(),
                         dtype=torch.float32, device=engine.device).requires_grad_(True)
    wo = torch.as_tensor(np.tile(np.concatenate([[spec.example_init], spec.scenario.init_state]), (B, 1, 1)),
                         dtype=torch.float32, device=engine.device).permute(1, 2, 0).contiguous()
    oc = torch.zeros((pr.C - 1, pr.H, 2, B), device=engine.device, requires_grad=True)
    plan, _, _ = torch.ops.ocd_b200.solve(wo, wr, None, oc, T.pack_params(pr))
    with pytest.raises(RuntimeError, match="other_controls"):
        plan.sum().backward()


def test_gradient_step_lowers_a_plan_matching_loss(engine):
    """A small step against the gradient of ||plan(w) - target||^2 lowers it by what the gradient predicts."""
    H, Cc = 5, 2
    op, batch, _ = _problem(H, Cc, 3, 0, False, 100, 0.1, 64, seed=12)
    w_full = batch["weights"][batch["weight_idx"]]
    ref, ref64, cond_u, _ = solve_conditioning(op, batch["world"], w_full)
    keep = np.nonzero((cond_u < 1e-6) & (ref["best"] == ref64["best"]))[0][:16]
    p = _pp(op, ocd.MATH_PRECISE)
    dev = engine.device
    world = torch.as_tensor(batch["world"][keep], device=dev).permute(1, 2, 0).contiguous()
    w0 = torch.as_tensor(w_full[keep], device=dev).t().contiguous()
    target = torch.as_tensor(ref["plan"][keep] + 0.05, device=dev).permute(1, 2, 0)

    def loss_of(w):
        plan, _, _ = torch.ops.ocd_b200.solve(world, w, None, None, T.pack_params(p))
        return ((plan - target) ** 2).sum()
    wg = w0.clone().requires_grad_(True)
    L0 = loss_of(wg)
    g, = torch.autograd.grad(L0, wg)
    step = 1e-3 * g / g.norm()
    with torch.no_grad():
        L1 = loss_of(w0 - step)
    predicted = -float((g * step).sum())
    actual = float(L1 - L0.detach())
    assert actual < 0 and 0.7 <= actual / predicted <= 1.3, (actual, predicted)
