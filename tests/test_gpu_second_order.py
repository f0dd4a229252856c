"""The kernels' second derivatives against an exact autodiff reference (oracle/autodiff64.py).

Every second-order kernel -- the feature Hessian (hyper-dual numbers, k_feature_hessian), the feature Jacobian, the
SGD solve VJP (vjp_hvp and grad_and_tangent through n_iter iterations) and the implicit-function VJP -- is compared
on every problem of its batch with the same derivative taken exactly by torch.func in float64.  There is no
differencing step, so no truncation error and no kink to skip.  The rule for an element is

    |gpu - ref64| <= 4 |ref32 - ref64| + atol * scale

with ref32 the same reference run in float32 (what float32 rounding loses on that problem), scale the maximum of
|ref64| over the matrix or vector, and atol for the kernels' different operation order.  Problems whose rollout comes
within 1e-5 of a branch decision (branch_margin) are left out; they may be at most 2 % of a batch.  Where a scale has a
floor, the test says why next to it.

The inputs (tests/second_order_cases.py) switch every curvature term on: the robot inside an other car's bump support,
inside the fence ramp on both sides, the speed feature under and over its bound, headings off pi/2, controls exactly
on the clip limits and beyond them.  Each test asserts that its inputs are not vacuous.

Worst (|gpu - ref64| - 4 |ref32 - ref64|) / scale seen on a B200, and the atol each test allows:
    feature Hessian, H <= 5 / 16 / 64     5.4e-5 / 1.5e-4 / 2.9e-4                        1e-4 / 2e-4 / 4e-4
    feature Jacobian, precise / fast      1.8e-5 / 1.9e-4                                  5e-5 / 4e-4
    phi_sum, precise / fast               4.0e-6 / 1.8e-4                                  2e-5 / 4e-4
    SGD solve VJP                         2.3e-4                                           4e-4
    implicit VJP (cond <= 1e5)            2.3e-6, plus cond 2^-24                          2e-5
    implicit VJP's residual               1.2e-5 of sum_k |w_k| max |d phi_k / du|          3e-5
    LocalCIOC.trajectory_terms            8.7e-8                                           2e-6
At H = 64 the Hessian's atol is 5x tighter than the 2e-3 of the difference-based test, not 10x: over 64 float32 steps
the kernel's operation order (libdevice sin / cos, reciprocals instead of divisions, FMA contraction) moves the
fence's curvature near the ramp's start by ~3e-4 of the matrix's largest entry, while a float32 CPU run of the
reference happens to stay closer to float64 there.  In fast math the SGD VJP's reference is taken along the GPU's own
stored iterates (their MUFU error is where the derivative is taken, not an error of the reverse pass).

Host time of the reference on the B200 machine (whole file 46 s of test time): the feature shapes 18 s in all (5.8 s at H = 64,
C = 8; 4.0 s at H = 64, C = 3; 4.7 s at H = 1, most of it the first use of torch.func), the solve VJPs 22 s (at most
2.0 s per case, fast math's reference along the GPU's iterates included), the implicit VJPs 4.7 s, LocalCIOC 0.4 s.
"""
import ctypes as C

import numpy as np
import pytest
import torch

import oracle as O
from oracle.autodiff64 import Reference

pytestmark = pytest.mark.gpu

import l4dc_mpc_ocd_b200 as ocd            # noqa: E402

from test_gpu_parity import _pp           # noqa: E402
from second_order_cases import (FEATURE_SHAPES, IVJP_SHAPES, VJP_CASES, feature_case, make_inputs,  # noqa: E402
                                params, vjp_case)

N = ocd._native

MARGIN = 1e-5                 # branch decisions closer than this to their threshold are not compared
ATOL = {"hess": {1: 1e-4, 2: 1e-4, 5: 1e-4, 16: 2e-4, 64: 4e-4}, "jac": {ocd.MATH_PRECISE: 5e-5, ocd.MATH_FAST: 4e-4}, "phi": {ocd.MATH_PRECISE: 2e-5,
        ocd.MATH_FAST: 4e-4}, "vjp": {ocd.MATH_PRECISE: 4e-4, ocd.MATH_FAST: 4e-4}, "ivjp": 2e-5, "residual": 3e-5,
        "cioc": 2e-6}
COND_MAX = 1e5
def excess(gpu, r64, r32, axes, floor=0.0):
    """(|gpu - ref64| - 4 |ref32 - ref64|) / scale per element, scale the maximum of |ref64| over `axes` (one matrix or
    vector) and at least `floor` (broadcast against it)."""
    gpu, r64, r32 = (np.asarray(a, np.float64) for a in (gpu, r64, r32))
    s = np.maximum(np.abs(r64).max(axis=axes, keepdims=True), floor)
    return (np.abs(gpu - r64) - 4 * np.abs(r32 - r64)) / np.where(s > 0, s, np.finfo(np.float64).tiny)


def checked(margin, B):
    """Problems far enough from every branch decision; the rest may be at most 2 % of the batch."""
    keep = margin >= MARGIN
    assert (~keep).sum() <= 0.02 * B, ((~keep).sum(), B)
    return keep


def report(name, worst):
    print(f"\n[second-order] {name}: worst normalised excess {worst:.3e}")


def nonzero_share(a, axes):
    """Share of problems on which `a` (leading axis: problem) is not identically zero."""
    return (np.abs(a) > 0).any(axis=axes).mean()


# ---- a, b: feature Hessian and Jacobian ---------------------------------------------------------------------------
_REF_CACHE = {}


def feature_refs(shape):
    """-> (op, inputs, hess64, hess32, jac64, jac32, phi64, phi32, margin), cached per shape."""
    if shape not in _REF_CACHE:
        op, inp = feature_case(*shape)
        out = [op, inp]
        for attr in ("batch_feature_hessian", "batch_feature_jacobian", "batch_phi_sum"):
            for dt in (torch.float64, torch.float32):
                out.append(getattr(Reference(op, dt), attr)(inp["world"], inp["u"], inp["oc"]))
        out.append(Reference(op).batch_branch_margin(inp["world"], inp["u"], inp["oc"]))
        _REF_CACHE[shape] = out
    return _REF_CACHE[shape]


@pytest.mark.parametrize("shape", FEATURE_SHAPES)
def test_feature_hessian_vs_autodiff(engine, shape):
    """ocd_feature_hessian_batch: every feature, both triangles, against hessian_u with one-hot weights."""
    op, inp, h64, h32, j64, *_, margin = feature_refs(shape)
    B, n = len(inp["world"]), 2 * op.H
    for k in range(op.K):                                             # every curvature term is exercised
        assert nonzero_share(h64[:, k], (1, 2)) >= 0.2, (k, nonzero_share(h64[:, k], (1, 2)))
    hes = engine.feature_hessian(_pp(op, ocd.MATH_PRECISE), inp["world"], inp["u"], other_controls=inp["oc"]).cpu().numpy()
    assert hes.shape == (B, op.K, n, n)
    assert np.array_equal(hes, hes.transpose(0, 1, 3, 2))
    keep = checked(margin, B)
    # A matrix that is zero in exact arithmetic can carry float32 cancellation noise, with ref32 blind to it: at H = 1
    # the fence past its ramp has T = F1 / (F1 + F2) with F2 = 0, whose derivatives cancel only in exact arithmetic;
    # one problem read gpu 1.7e-13, ref64 -2.5e-22, ref32 exactly 0.  So each matrix's scale is at least 1e-4 of the
    # same feature's largest first derivative (its own accumulator: another feature's size never enters).
    ex = excess(hes, h64, h32, (2, 3), floor=1e-4 * np.abs(j64).max(axis=2)[..., None, None])
    b, k, i, j = np.unravel_index(np.argmax(np.where(keep[:, None, None, None], ex, -np.inf)), ex.shape)
    print(f"\nworst at problem {b} feature {k} ({i}, {j}): gpu {hes[b, k, i, j]:.9e} ref64 {h64[b, k, i, j]:.9e} "
          f"ref32 {h32[b, k, i, j]:.9e} scale {np.abs(h64[b, k]).max():.3e} margin {margin[b]:.2e}")
    ex = ex[keep]
    report(f"hess {shape}", ex.max())
    assert ex.max() <= ATOL["hess"][op.H], ex.max()


@pytest.mark.parametrize("mode", [ocd.MATH_PRECISE, ocd.MATH_FAST])
@pytest.mark.parametrize("shape", FEATURE_SHAPES)
def test_feature_jacobian_vs_autodiff(engine, shape, mode):
    """ocd_feature_jacobian_batch: phi_sum and jac, both math modes, on the Hessian test's inputs."""
    op, inp, _, _, j64, j32, p64, p32, margin = feature_refs(shape)
    B = len(inp["world"])
    for k in range(op.K):
        assert nonzero_share(j64[:, k], (1,)) >= 0.2, k
    phi, jac = engine.feature_jacobian(_pp(op, mode), inp["world"], inp["u"], other_controls=inp["oc"])
    phi, jac = phi.cpu().numpy(), jac.cpu().numpy().reshape(B, op.K, -1)
    keep = checked(margin, B)
    # Fast math's sin / cos (MUFU) err by up to 2^-21.4 absolutely: an error of the state that every feature shares.
    # Next to where a feature switches on, its value and derivatives are tiny and steep in the state -- the fence at
    # its ramp start (exp(-1 / (shape q)), small q), the bump at its support edge -- so that error is a large part of
    # them: at H = 1 one fence read phi 1.3885e-18 against 1.3860e-18 in float64 (the problem's largest feature 0.59),
    # at H = 5 one collision feature 2.136e-31 against 2.124e-31.  In fast math a row's scale is therefore at least
    # 1e-4 of the problem's largest entry; precise math, the same kernel code with libdevice functions, is held to
    # each row's and each feature's own scale.
    fast = mode == ocd.MATH_FAST
    ej = excess(jac, j64, j32, (2,), floor=1e-4 * np.abs(j64).max(axis=(1, 2))[:, None, None] if fast else 0.0)[keep]
    ep = excess(phi[..., None], p64[..., None], p32[..., None], (2,),
                floor=1e-4 * np.abs(p64).max(axis=1)[:, None, None] if fast else 0.0)[keep]
    report(f"jac {shape} mode={mode}", ej.max())
    report(f"phi {shape} mode={mode}", ep.max())
    assert ej.max() <= ATOL["jac"][mode], ej.max()
    assert ep.max() <= ATOL["phi"][mode], ep.max()


# ---- c: sentinel bands ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [1, 127, 129, 1000])
def test_feature_outputs_stay_in_bounds(engine, B):
    """phi_sum, jac and hess are windows inside sentinel-filled buffers at ragged batch sizes, H = 64, C = 8, L = 4:
    the guard bands must survive and every element must be written.  The Hessian (K 2H 2H B floats) is checked up to
    B = 129."""
    op = params(64, 8, 4, 1)
    inp = make_inputs(op, B, seed=B, Bo=B)
    p = _pp(op, ocd.MATH_PRECISE).c_struct()
    dev = engine.device
    world = torch.as_tensor(inp["world"], device=dev).permute(1, 2, 0).contiguous()
    u = torch.as_tensor(inp["u"], device=dev).permute(1, 2, 0).contiguous()
    oc = torch.as_tensor(inp["oc"], device=dev).permute(1, 2, 3, 0).contiguous()
    n = 2 * op.H
    G, SENT = 4096, 12345.0
    sizes = dict(phi=op.K * B, jac=op.K * n * B)
    if B <= 129:
        sizes["hess"] = op.K * n * n * B
    bufs = {k: torch.full((m + 2 * G,), SENT, dtype=torch.float32, device=dev) for k, m in sizes.items()}
    win = {k: bufs[k][G:G + m] for k, m in sizes.items()}
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    ptr = lambda t: C.c_void_p(t.data_ptr())                                     # noqa: E731
    N.check(N.lib.ocd_feature_jacobian_batch(C.addressof(p), ptr(world), ptr(u), ptr(oc), B, ptr(win["phi"]),
                                             ptr(win["jac"]), B, stream), "ocd_feature_jacobian_batch")
    if "hess" in win:
        N.check(N.lib.ocd_feature_hessian_batch(C.addressof(p), ptr(world), ptr(u), ptr(oc), B, ptr(win["hess"]), B,
                                                stream), "ocd_feature_hessian_batch")
    torch.cuda.synchronize()
    for k, m in sizes.items():
        assert (bufs[k][:G] == SENT).all() and (bufs[k][G + m:] == SENT).all(), k
        assert (win[k] != SENT).all(), k
        assert torch.isfinite(win[k]).all(), k


# ---- d: the SGD solve VJP at short budgets ------------------------------------------------------------------------
_VJP_CACHE = {}


def vjp_refs(shape, n_iter, best):
    key = (shape, n_iter, tuple(best))
    if key not in _VJP_CACHE:
        op, inp, pbar = vjp_case(shape, n_iter)
        r = [Reference(op, dt).batch_sgd_vjp(inp["world"], inp["w"], best, n_iter, pbar, inp["oc"])
             for dt in (torch.float64, torch.float32)]
        _VJP_CACHE[key] = r
    return _VJP_CACHE[key]


def _soa(engine, inp):
    dev = engine.device
    world = torch.as_tensor(inp["world"], device=dev).permute(1, 2, 0).contiguous()
    w = torch.as_tensor(inp["w"], device=dev).t().contiguous()
    oc = None if inp["oc"] is None else torch.as_tensor(inp["oc"], device=dev).permute(1, 2, 3, 0).contiguous()
    return world, w, oc


def _solve_vjp_raw(engine, p, world, w, oc, Bo, best, pb):
    """ocd_solve_vjp_batch with a workspace of our own -> (weights_bar [B, K], world_bar [B, C, 4], the stored
    iterates u^0 .. u^{N-1} [B, N, 2H])."""
    B, dev = world.shape[-1], engine.device
    ps = p.c_struct()
    nb = C.c_size_t(0)
    N.check(N.lib.ocd_solve_vjp_workspace_bytes(C.addressof(ps), B, C.byref(nb)), "workspace")
    ws = torch.empty((nb.value // 4,), dtype=torch.float32, device=dev)
    wb = torch.empty((p.K, B), dtype=torch.float32, device=dev)
    xb = torch.empty((p.C, 4, B), dtype=torch.float32, device=dev)
    ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())              # noqa: E731
    N.check(N.lib.ocd_solve_vjp_batch(C.addressof(ps), ptr(world), ptr(oc), Bo, ptr(w), B, None, None, ptr(best),
                                      ptr(pb), ptr(wb), ptr(xb), ptr(ws) if nb.value else None, nb.value, B,
                                      C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "ocd_solve_vjp_batch")
    its = ws.view(p.n_iter, 2 * p.H, B).permute(2, 0, 1).cpu().numpy()
    return wb.t().cpu().numpy(), xb.permute(2, 0, 1).cpu().numpy(), its


@pytest.mark.parametrize("mode", [ocd.MATH_PRECISE, ocd.MATH_FAST])
@pytest.mark.parametrize("shape,n_iter", [(s, n) for s, ns in VJP_CASES for n in ns])
def test_solve_vjp_vs_autodiff(engine, shape, n_iter, mode):
    """ocd_solve_vjp_batch: weights_bar and every car's world_bar, every problem, against torch.func.vjp of sgd_plan
    for the start the GPU picked."""
    op, inp, pbar = vjp_case(shape, n_iter)
    B = len(inp["world"])
    p = _pp(op, mode)
    world, w, oc = _soa(engine, inp)
    Bo = 0 if oc is None else B
    if n_iter == 0:
        nb, ps = C.c_size_t(1), p.c_struct()
        N.check(N.lib.ocd_solve_vjp_workspace_bytes(C.addressof(ps), B, C.byref(nb)), "workspace")
        assert nb.value == 0
    # ocd_solve_batch refuses precise math at H = 64 with seven other cars and six starts (its shared-memory slab does
    # not fit); the VJP takes the winning start as an input, so there the fast forward's winner is differentiated
    fwd_p = _pp(op, ocd.MATH_FAST) if op.H == 64 else p
    fwd = engine.solve_soa(fwd_p, world, w, B, None, oc, Bo)
    pb = torch.as_tensor(pbar, device=engine.device).permute(1, 2, 0).contiguous()
    wb, xb, its = _solve_vjp_raw(engine, p, world, w, oc, Bo, fwd["best"], pb)
    best = fwd["best"].cpu().numpy()
    (w64, x64, margin), (w32, x32, _) = vjp_refs(shape, n_iter, best)
    if mode == ocd.MATH_FAST and n_iter > 0:
        # the fast forward's iterates carry MUFU error; the reverse pass is exact along them, so the reference is
        # taken along the same iterates (margins still from the float64 run, a few ulps away)
        w64, x64 = Reference(op).batch_sgd_vjp_along(inp["world"], inp["w"], best, its, pbar, inp["oc"])
        w32, x32 = Reference(op, torch.float32).batch_sgd_vjp_along(inp["world"], inp["w"], best, its, pbar,
                                                                    inp["oc"])
    if n_iter == 0:
        # the plan is the start: only the extra-init starts (a0 = friction v0^2) depend on anything, the robot's speed
        assert np.all(wb == 0.0)
        rest = xb.copy()
        rest[:, 0, 2] = 0.0
        assert np.all(rest == 0.0)
        assert np.array_equal(xb[:, 0, 2] != 0.0, best >= 3)
    else:
        for k in range(op.K):
            assert nonzero_share(w64[:, k], ()) >= 0.2, k
        assert nonzero_share(x64[:, 1:], (1, 2)) >= 0.2
    keep = checked(margin, B)
    ew = excess(wb, w64, w32, (1,))[keep]
    ex = excess(xb.reshape(B, -1), x64.reshape(B, -1), x32.reshape(B, -1), (1,))[keep]
    report(f"vjp {shape} n_iter={n_iter} mode={mode}", max(ew.max(), ex.max()))
    assert ew.max() <= ATOL["vjp"][mode], ew.max()
    assert ex.max() <= ATOL["vjp"][mode], ex.max()


# ---- e: the implicit-function VJP at the GPU's own L-BFGS plan ---------------------------------------------------


@pytest.mark.parametrize("shape", IVJP_SHAPES)
def test_solve_implicit_vjp_vs_autodiff(engine, shape):
    """ocd_solve_implicit_vjp_batch against implicit_vjp at the plan the GPU's L-BFGS returned.  Problems with
    cond(H_AA) <= 1e5 are compared, with cond 2^-24 added to atol; a NaN row must fall on a problem the reference
    finds singular or ill-conditioned.  residual must be max |grad_u| over the clip-box controls."""
    H, Cc, L, other_mode, Bo = shape
    B = 128
    op = params(H, Cc, L, other_mode, n_iter=40, optimizer=1)
    inp = make_inputs(op, B, seed=3000 + 11 * H + Cc, Bo=B if Bo == "B" else Bo, controls=False)
    p = _pp(op, ocd.MATH_PRECISE)
    p.optimizer = ocd.OPT_LBFGS
    world, w, oc = _soa(engine, inp)
    Bo_ = 0 if oc is None else oc.shape[-1]
    fwd = engine.solve_soa(p, world, w, B, None, oc, Bo_)
    pbar = np.random.default_rng(H).normal(size=(B, H, 2)).astype(np.float32)
    pb = torch.as_tensor(pbar, device=engine.device).permute(1, 2, 0).contiguous()
    out = engine.solve_implicit_vjp_soa(p, world, w, B, fwd["plan"], pb, None, oc, Bo_, residual=True)
    plan = fwd["plan"].permute(2, 0, 1).cpu().numpy()
    wb = out["weights_bar"].t().cpu().numpy()
    xb = out["world_bar"].permute(2, 0, 1).cpu().numpy().reshape(B, -1)
    res = out["residual"].cpu().numpy()
    r64, r32 = Reference(op), Reference(op, torch.float32)
    w64, x64, cond = r64.implicit_vjp(inp["world"], inp["w"], plan, pbar, inp["oc"])
    w32, x32, _ = r32.implicit_vjp(inp["world"], inp["w"], plan, pbar, inp["oc"])
    margin = r64.batch_branch_margin(inp["world"], plan, inp["oc"])
    nan = ~np.isfinite(wb).all(1) | ~np.isfinite(xb).all(1)
    assert np.all(cond[nan] > COND_MAX), cond[nan]
    well = (cond <= COND_MAX) & checked(margin, B)
    assert not nan[cond <= COND_MAX].any()
    assert well.sum() >= 16, well.sum()
    for k in range(op.K):
        assert nonzero_share(w64[well][:, k], ()) >= 0.2, k
    assert nonzero_share(x64[well][:, 1:], (1, 2)) >= 0.2
    tol = (ATOL["ivjp"] + cond * 2.0 ** -24)[:, None]
    ew = (excess(wb, w64, w32, (1,)) - tol)[well]
    ex = (excess(xb, x64.reshape(B, -1), x32.reshape(B, -1), (1,)) - tol)[well]
    report(f"ivjp {shape} ({well.sum()} of {B} compared)", max(ew.max(), ex.max()) + ATOL["ivjp"])
    assert ew.max() <= 0 and ex.max() <= 0, (ew.max(), ex.max())
    # residual: max |dR/du| over the controls inside the clip box, at the plan.  A converged plan's gradient is a sum
    # of cancelling terms, so its rounding is relative to their size: sum_k |w_k| max |d phi_k / du|.
    u = plan.reshape(B, -1).astype(np.float64)
    act = np.ones_like(u, bool)
    act[:, 0::2] = (u[:, 0::2] >= -8.0) & (u[:, 0::2] <= 4.0)
    act[:, 1::2] = np.abs(u[:, 1::2]) <= 4.0
    g64 = r64.batch_reward(inp["world"], plan, inp["w"], inp["oc"])[1]
    g32 = r32.batch_reward(inp["world"], plan, inp["w"], inp["oc"])[1]
    terms = (np.abs(inp["w"]) * np.abs(r64.batch_feature_jacobian(inp["world"], plan, inp["oc"])).max(2)).sum(1)
    res64, res32 = (np.where(act, np.abs(g), 0.0).max(1) for g in (g64, g32))
    er = ((np.abs(res - res64) - 4 * np.abs(res32 - res64)) / np.maximum(terms, 1e-30))[checked(margin, B)]
    report(f"residual {shape}", er.max())
    assert er.max() <= ATOL["residual"], er.max()


# ---- f: LocalCIOC's assembly of windows -------------------------------------------------------------------------
@pytest.mark.parametrize("split", [False, True])
def test_local_cioc_terms_vs_autodiff(split):
    """LocalCIOC.trajectory_terms on a planned trajectory: G [K, 2T] and Hm [K, 2T, 2T] against the reference evaluated
    window by window.  Column c is control c of the trajectory; it comes from the window that starts at
    min(c // 2, T - H) (split_traj: (c // 2H) H) at row c - 2 start."""
    from l4dc_mpc_ocd_b200.interact_drive.reward_design import LocalCIOC
    from test_gpu_ioc import _drive
    world, car, traj, _ = _drive(T=10)
    T, H, me = len(traj), car.planner.horizon, car.index
    cioc = LocalCIOC(car, weight_norm=1., split_traj=split)
    G, Hm = cioc.trajectory_terms(traj)
    op = O.OracleParams(H=H, C=2, lane_x=tuple(world.lane_medians()), num_lanes=int(car.num_lanes), other_mode=0,
                        dt=world.dt, friction=float(car.friction), target_speed=float(car.target_speed))
    starts = list(range(0, T - H + 1, H)) if split else list(range(T - H + 1))
    st = np.stack([np.stack([np.asarray(s, np.float32).reshape(4) for s in traj[i][0]]) for i in starts])
    st = st[:, [me] + [c for c in range(st.shape[1]) if c != me]]
    u = np.stack([np.stack([np.asarray(traj[i + j][1][me], np.float32).reshape(2) for j in range(H)]) for i in starts])
    refs = []
    for dt in (torch.float64, torch.float32):
        r = Reference(op, dt)
        refs.append((r.batch_feature_jacobian(st, u), r.batch_feature_hessian(st, u)))
    margin = Reference(op).batch_branch_margin(st, u)
    assert np.all(margin >= MARGIN), margin
    K = op.K
    G_ref, H_ref = [np.zeros((K, 2 * T)) for _ in refs], [np.zeros((K, 2 * T, 2 * T)) for _ in refs]
    for c in range(2 * T):
        wi = (c // (2 * H)) if split else min(c // 2, T - H)
        i = starts[wi]
        for (jac, hes), Gr, Hr in zip(refs, G_ref, H_ref):
            Gr[:, c] = jac[wi][:, c - 2 * i]
            Hr[:, c, 2 * i:2 * i + 2 * H] = hes[wi][:, c - 2 * i]
    assert G.shape == G_ref[0].shape and Hm.shape == H_ref[0].shape
    assert np.abs(H_ref[0]).max() > 0
    eg = excess(G, G_ref[0], G_ref[1], (1,))
    eh = excess(Hm, H_ref[0], H_ref[1], (1, 2))
    report(f"cioc split={split}", max(eg.max(), eh.max()))
    assert eg.max() <= ATOL["cioc"] and eh.max() <= ATOL["cioc"], (eg.max(), eh.max())
