"""ocd_episode_vjp_batch, Engine.episodes_vjp_soa, the autograd formula of torch.ops.ocd_b200.episodes and
MPC_ORD.eval_weights_grad on the GPU.

The independent route is the f64 CPU oracle: whole episodes differenced in random directions of the planning
weights, the robot's initial state and the true weights.  Full-budget episodes are checked on the worlds the parity
tests' probe (episode_conditioning) finds reproducible and whose winning starts the f64 oracle reproduces at every
step; at two iterations and three steps every world is checked."""
import ctypes as C
import dataclasses

import numpy as np
import pytest
import torch

import oracle as O

pytestmark = pytest.mark.gpu

import l4dc_mpc_ocd_b200 as ocd            # noqa: E402
from l4dc_mpc_ocd_b200 import torch_ops as TO    # noqa: E402

from test_gpu_parity import MODES, _pp, _sc, episode_conditioning    # noqa: E402

N = ocd._native

# (scenario, horizon, extra-init starts, control steps): finite_horizon, local_opt, replanning (two fixed-plan cars,
# known controls, the teleport), H = 6 with six starts and 200 iterations, and H = 15 at lr 0.02 (an episode runs it on
# the runtime-horizon segmented kernels, not on the solve's compile-time H = 15 kernels)
SHAPES = [("finite_horizon", 5, False, 15), ("local_opt", 5, False, 15), ("replanning", 5, False, 20),
          ("finite_horizon", 6, True, 15), ("finite_horizon", 15, False, 15)]
SHORT = [s for s in SHAPES if s[1] <= 6]


def _spec(name, H, extra, n_iter=None):
    spec = O.scenario_params(name, horizon=H, extra_inits=extra)
    op = spec.params
    if n_iter is not None:
        op = dataclasses.replace(op, n_iter=n_iter)
    if H > 8:                      # lr 0.1 is too long a step for long horizons
        op = dataclasses.replace(op, lr=0.02)
    return dataclasses.replace(spec, params=op)


def _batch(spec, B, seed):
    """B worlds around the scenario's example state, B // 4 candidate weight vectors near the designer's (indexed),
    and -- replanning -- the car that teleports in each."""
    rng = np.random.default_rng(seed)
    K, Cc = spec.params.K, spec.params.C
    ri = np.tile(spec.example_init.astype(np.float32), (B, 1))
    ri[:, 0] += rng.uniform(-0.03, 0.03, B).astype(np.float32)
    ri[:, 1] += rng.uniform(-0.04, 0.04, B).astype(np.float32)
    ri[:, 2] += rng.uniform(-0.08, 0.08, B).astype(np.float32)
    wt = (spec.designer_weights / np.linalg.norm(spec.designer_weights)).astype(np.float32)
    nc = max(1, B // 4)
    cand = wt[None] + 0.05 * rng.normal(size=(nc, K))
    cand = (cand / np.linalg.norm(cand, axis=1, keepdims=True)).astype(np.float32)
    widx = (np.arange(B) % nc).astype(np.int32)
    ul = rng.integers(1, Cc, B).astype(np.int32) if spec.scenario.critical_t > 0 else None
    return ri, cand, wt, widx, ul


def _dev(engine, ri, cand, wt, widx, ul):
    d = engine.device
    return (torch.as_tensor(ri.T.copy(), device=d), torch.as_tensor(cand.T.copy(), device=d), torch.as_tensor(wt, device=d),
            torch.as_tensor(widx, device=d), None if ul is None else torch.as_tensor(ul, device=d))


def _run(engine, p, sc, T, ri, cand, wt, widx, ul, rbar=None):
    """Forward with trace, then the VJP; -> (forward dict, per-world rows as float64 [B, ...])."""
    ris, w, tw, idx, ult = _dev(engine, ri, cand, wt, widx, ul)
    fwd = engine.episodes_soa(p, sc, ris, w, w.shape[1], tw, T, weight_idx=idx, unlucky_idx=ult, trace=True)
    rb = torch.ones_like(fwd["returns"]) if rbar is None else torch.as_tensor(rbar, device=engine.device)
    g = engine.episodes_vjp_soa(p, sc, w, w.shape[1], tw, T, fwd["states"], fwd["best"], fwd["controls"], rb, idx)
    return fwd, {k: v.t().cpu().numpy().astype(np.float64) for k, v in g.items()}


def _ret64(spec, T, ri, wp, wt, ul):
    return float(O.episode(spec.params, spec.scenario, ri, wp, wt, T, unlucky_idx=ul, dtype=np.float64)["ret"])


def _compare(spec, T, worlds, ri, wfull, wt, ul, g, rng, h, limit=None):
    """Random directions over the planning weights, the robot's initial state and the true weights, against central
    differences of the f64 oracle at h and h / 2.  -> (relative errors of the checked worlds, number at a kink)."""
    errs, skipped = [], 0
    for b in worlds:
        if limit is not None and len(errs) >= limit:
            break
        dw, dt = rng.normal(size=wfull.shape[1]), rng.normal(size=wfull.shape[1])
        dx = rng.normal(size=4) * np.array([0.02, 0.02, 0.1, 0.05])
        u = 0 if ul is None else int(ul[b])
        x64, w64, t64 = ri[b].astype(np.float64), wfull[b].astype(np.float64), wt.astype(np.float64)

        def q(hh):
            return (_ret64(spec, T, x64 + hh * dx, w64 + hh * dw, t64 + hh * dt, u)
                    - _ret64(spec, T, x64 - hh * dx, w64 - hh * dw, t64 - hh * dt, u)) / (2 * hh)
        q1, q2 = q(h), q(h / 2)
        scale = max(abs(q1), 1e-2)
        if abs(q1 - q2) > 1e-3 * scale:           # a kink inside the interval: the quotient means nothing there
            skipped += 1
            continue
        got = float(g["plan_weights_bar"][b] @ dw + g["robot_init_bar"][b] @ dx + g["true_weights_bar"][b] @ dt)
        errs.append(abs(got - q2) / scale)
    return np.asarray(errs), skipped


@pytest.mark.parametrize("mode,_n", MODES)
@pytest.mark.parametrize("name,H,extra,T", SHAPES)
def test_episode_vjp_vs_oracle_differences(engine, mode, _n, name, H, extra, T):
    spec = _spec(name, H, extra)
    p, sc = _pp(spec.params, mode), _sc(spec.scenario)
    B = 160
    ri, cand, wt, widx, ul = _batch(spec, B, seed=17 * H + len(name))
    fwd, g = _run(engine, p, sc, T, ri, cand, wt, widx, ul)
    finite = np.all([np.isfinite(v).all(axis=1) for v in g.values()], axis=0)
    wfull = cand[widx]
    _, spread = episode_conditioning(spec, ri, wfull, wt, T, ul)
    # Where the planner's SGD map is locally expansive (spectral radius of I + lr dG/du up to ~10 on some H = 15 worlds
    # at lr 0.02) the derivative through 100 iterations grows like rho^100 and overflows float32.  Such a world's return
    # amplifies ulp-sized noise just as much, so the oracle's own probe finds it irreproducible: a gradient may only be
    # non-finite there.
    assert not np.any(~finite & (spread < 1e-5)), np.nonzero(~finite & (spread < 1e-5))[0]
    best = fwd["best"].cpu().numpy().T                                   # [B, T]
    well = []
    for b in np.nonzero(spread < 1e-5)[0]:
        o = O.episode(spec.params, spec.scenario, ri[b].astype(np.float64), wfull[b].astype(np.float64),
                      wt.astype(np.float64), T, unlucky_idx=0 if ul is None else int(ul[b]), dtype=np.float64)
        if np.array_equal(o["best"], best[b]):
            well.append(b)
    rng = np.random.default_rng(H + T)
    # a short step: at H = 15 many returns curve strongly on the scale of 1e-5 (the quotients at 1e-5 and 5e-6 disagree
    # on half the reproducible worlds, at 1e-7 and 5e-8 on a thirtieth), and f64 leaves the quotients enough digits
    errs, skipped = _compare(spec, T, well, ri, wfull, wt, ul, g, rng, 1e-7, limit=40)
    print(f"{name} H={H} T={T} mode={mode}: {int((~finite).sum())} non-finite, {len(well)} reproducible, "
          f"{len(errs)} checked, {skipped} at a kink, "
          f"median {np.median(errs):.2e}, worst {errs.max():.2e}")
    assert len(errs) >= 12, (len(well), len(errs), skipped)
    assert len(errs) >= 0.8 * (len(errs) + skipped), (len(errs), skipped)
    assert np.median(errs) <= 1e-3
    assert np.mean(errs <= 2e-2) >= 0.95, np.sort(errs)[-5:]


@pytest.mark.parametrize("mode,_n", MODES)
@pytest.mark.parametrize("name,H,extra,T", SHAPES)
def test_short_budget_every_world(engine, mode, _n, name, H, extra, T):
    """Two SGD iterations and three control steps amplify nothing: every world is checked (bar a kink inside the
    differencing interval, or a winning start the f64 oracle does not reproduce)."""
    spec = _spec(name, H, extra, n_iter=2)
    p, sc = _pp(spec.params, mode), _sc(spec.scenario)
    B, T = 200, 3
    ri, cand, wt, widx, ul = _batch(spec, B, seed=5 + H)
    fwd, g = _run(engine, p, sc, T, ri, cand, wt, widx, ul)
    wfull = cand[widx]
    best = fwd["best"].cpu().numpy().T
    same = []
    for b in range(B):
        o = O.episode(spec.params, spec.scenario, ri[b].astype(np.float64), wfull[b].astype(np.float64),
                      wt.astype(np.float64), T, unlucky_idx=0 if ul is None else int(ul[b]), dtype=np.float64)
        if np.array_equal(o["best"], best[b]):
            same.append(b)
    errs, skipped = _compare(spec, T, same, ri, wfull, wt, ul, g, np.random.default_rng(H), 1e-6)
    assert skipped + (B - len(same)) <= 0.03 * B, (skipped, B - len(same))
    assert errs.max() <= 2e-3, np.sort(errs)[-5:]


def _planner_other_controls(p, spec):
    """The planner's model of the scripted cars in an episode as solve_soa's other_controls [C-1][H][2][1]: a fixed-plan
    car's plan replayed from index 0, then its control; zero for the others."""
    oc = np.zeros((p.C - 1, p.H, 2, 1), np.float32)
    s = spec.scenario
    for j in range(p.C - 1):
        if s.kind[j] == 1:
            for t in range(p.H):
                oc[j, t, :, 0] = s.plan[j][t] if t < len(s.plan[j]) else s.control[j]
    return oc


@pytest.mark.parametrize("mode,_n", MODES)
@pytest.mark.parametrize("name,H,extra,T", SHORT)
def test_composition_of_solve_vjps(engine, mode, _n, name, H, extra, T):
    """The episode VJP equals a host-side chain built from T x 2 one-hot Engine.solve_vjp_soa calls (the Jacobian of
    each applied control), the oracle's feature Jacobian and the simulator step's adjoint in float64."""
    spec = _spec(name, H, extra)
    p, sc = _pp(spec.params, mode), _sc(spec.scenario)
    B = 48
    ri, cand, wt, widx, ul = _batch(spec, B, seed=3 * H)
    fwd, g = _run(engine, p, sc, T, ri, cand, wt, widx, ul)
    dev = engine.device
    _, w, _, idx, _ = _dev(engine, ri, cand, wt, widx, ul)
    oc = torch.as_tensor(_planner_other_controls(p, spec), device=dev) if p.other_mode == 1 else None
    K = p.K
    J = np.zeros((T, 2, K + 4, B))
    for t in range(T):
        for c in range(2):
            pb = torch.zeros((p.H, 2, B), device=dev)
            pb[0, c] = 1.0
            o = engine.solve_vjp_soa(p, fwd["states"][t].contiguous(), w, w.shape[1], fwd["best"][t].contiguous(), pb,
                                     idx, oc, 1 if oc is not None else 0)
            J[t, c, :K] = o["weights_bar"].cpu().numpy()
            J[t, c, K:] = o["world_bar"][0].cpu().numpy()
    S = fwd["states"].cpu().numpy().astype(np.float64)        # [T][C][4][B]
    U = fwd["controls"].cpu().numpy().astype(np.float64)      # [T][2][B]
    dt, mu = p.dt, p.friction
    hdt2 = 0.5 * float(np.float32(dt * dt))
    op64 = spec.params
    for b in range(B):
        lam, wbar, tbar = np.zeros(4), np.zeros(K), np.zeros(K)
        for t in range(T - 1, -1, -1):
            x, y, v, th = S[t, 0, :, b]
            a, om = U[t, :, b]
            ac = min(max(a, -8.0), 4.0)
            dist = v * dt + hdt2 * (ac - mu * v * v)
            ld = np.cos(th) * lam[0] + np.sin(th) * lam[1]
            lt = hdt2 * ld + dt * lam[2]
            ub = np.array([lt if -8.0 <= a <= 4.0 else 0.0, dt * lam[3] if abs(om) <= 4.0 else 0.0])
            nl = np.array([lam[0], lam[1], lam[2] + dt * ld - 2 * mu * v * lt,
                           lam[3] + dist * (np.cos(th) * lam[1] - np.sin(th) * lam[0])])
            wbar += ub @ J[t, :, :K, b]
            nl += ub @ J[t, :, K:, b]
            phi, jac = O.features(op64, S[t, :, :, b], dtype=np.float64, jac=True)
            nl += wt.astype(np.float64) @ jac
            tbar += phi
            lam = nl
        for got, want in ((g["plan_weights_bar"][b], wbar), (g["robot_init_bar"][b], lam), (g["true_weights_bar"][b], tbar)):
            np.testing.assert_allclose(got, want, rtol=1e-5, atol=1e-5 * max(1.0, np.abs(want).max()), err_msg=f"world {b}")


def _raw(engine, p, sc, T, fwd, w, idx, tw, rb, ws_bytes, G=1024, SENT=12345.0):
    """ocd_episode_vjp_batch with every output and the workspace a window inside a sentinel-filled buffer."""
    B = rb.shape[0]
    dev = engine.device
    ps, ss = p.c_struct(), sc.c_struct()
    sizes = dict(wbar=p.K * B, rbar=4 * B, tbar=p.K * B, ws=ws_bytes // 4)
    bufs = {k: torch.full((n + 2 * G,), SENT, dtype=torch.float32, device=dev) for k, n in sizes.items()}
    win = {k: bufs[k][G:G + n] for k, n in sizes.items()}
    ptr = lambda t: C.c_void_p(t.data_ptr())
    rc = N.lib.ocd_episode_vjp_batch(C.addressof(ps), C.addressof(ss), ptr(w), w.shape[1],
                                     None if idx is None else ptr(idx), ptr(tw), T, ptr(fwd["states"]),
                                     ptr(fwd["best"]), ptr(fwd["controls"]), ptr(rb), ptr(win["wbar"]), ptr(win["rbar"]),
                                     ptr(win["tbar"]), ptr(win["ws"]), ws_bytes, B,
                                     C.c_void_p(torch.cuda.current_stream().cuda_stream))
    N.check(rc, "ocd_episode_vjp_batch")
    torch.cuda.synchronize()
    return bufs, win


def _ws_bytes(p, T, B):
    lo, full = C.c_size_t(0), C.c_size_t(0)
    ps = p.c_struct()
    N.check(N.lib.ocd_episode_vjp_workspace_bytes(C.addressof(ps), T, B, C.byref(lo), C.byref(full)))
    return lo.value, full.value


@pytest.mark.parametrize("name,H,extra,T", SHAPES)
def test_iterates_are_the_episodes_own(engine, monkeypatch, name, H, extra, T):
    """With the full workspace every step's iterates stay in it: u^N's first control is traj_controls[t] bit for bit,
    at every step, whichever form ran the forward episode, in both math modes."""
    spec = _spec(name, H, extra)
    B = 97
    ri, cand, wt, widx, ul = _batch(spec, B, seed=11 + H)
    for mode, forms in ((ocd.MATH_FAST, ("throughput", "latency", "wide", "tp", None)), (ocd.MATH_PRECISE, (None,))):
        p, sc = _pp(spec.params, mode), _sc(spec.scenario)
        ris, w, tw, idx, ult = _dev(engine, ri, cand, wt, widx, ul)
        lo, full = _ws_bytes(p, T, B)
        for form in forms:
            if form:
                monkeypatch.setenv("OCD_KERNEL_FORM", form)
            fwd = engine.episodes_soa(p, sc, ris, w, w.shape[1], tw, T, weight_idx=idx, unlucky_idx=ult, trace=True)
            monkeypatch.delenv("OCD_KERNEL_FORM", raising=False)
            _, win = _raw(engine, p, sc, T, fwd, w, idx, tw, torch.ones(B, device=engine.device), full)
            jac = T * 2 * (p.K + 4) * B
            its = win["ws"][jac:].view(T, p.n_iter + 1, p.H, 2, B)
            assert torch.equal(its[:, p.n_iter, 0], fwd["controls"]), (name, H, mode, form)


@pytest.mark.parametrize("name,H,extra,T,B", [("finite_horizon", 5, False, 15, 33), ("replanning", 5, False, 20, 1),
                                              ("finite_horizon", 6, True, 15, 130), ("local_opt", 5, False, 15, 4097),
                                              ("finite_horizon", 15, False, 15, 65)])
def test_workspace_sizes_agree_and_stay_in_bounds(engine, name, H, extra, T, B):
    """The minimum workspace (one step in flight), a ragged step group and the full workspace give bit-identical
    outputs; every output and the workspace sit inside sentinel-filled buffers whose guard bands must survive, and the
    windows are fully written."""
    spec = _spec(name, H, extra)
    spec = dataclasses.replace(spec, params=dataclasses.replace(spec.params, n_iter=12))
    p, sc = _pp(spec.params, ocd.MATH_FAST), _sc(spec.scenario)
    ri, cand, wt, widx, ul = _batch(spec, B, seed=B)
    ris, w, tw, idx, ult = _dev(engine, ri, cand, wt, widx, ul)
    fwd = engine.episodes_soa(p, sc, ris, w, w.shape[1], tw, T, weight_idx=idx, unlucky_idx=ult, trace=True)
    rb = torch.as_tensor(np.random.default_rng(B).normal(size=B), dtype=torch.float32, device=engine.device)
    lo, full = _ws_bytes(p, T, B)
    step = (full - lo) // (T - 1)
    G, SENT = 1024, 12345.0
    res = {}
    for label, nb in (("min", lo), ("ragged", lo + 3 * step + 4), ("full", full)):
        bufs, win = _raw(engine, p, sc, T, fwd, w, idx, tw, rb, nb, G, SENT)
        for k, buf in bufs.items():
            n = win[k].numel()
            assert (buf[:G] == SENT).all() and (buf[G + n:] == SENT).all(), (label, k)
            if label != "ragged" or k != "ws":
                assert (buf[G:G + n] != SENT).all(), (label, k)
        res[label] = {k: win[k].clone() for k in ("wbar", "rbar", "tbar")}
        assert all(torch.isfinite(v).all() for v in res[label].values())
    for label in ("ragged", "full"):
        for k in res["min"]:
            assert torch.equal(res["min"][k], res[label][k]), (label, k)


# ---- autograd -----------------------------------------------------------------------------------------------------
def _ep(ris, w, idx, tw, ult, p, sc, T):
    return torch.ops.ocd_b200.episodes(ris, w, idx, tw, ult, TO.pack_params(p), TO.pack_scenario(sc), T)


@pytest.mark.parametrize("name", ["finite_horizon", "replanning"])
def test_autograd_matches_the_engine(engine, name):
    spec = _spec(name, 5, False)
    p, sc = _pp(spec.params, ocd.MATH_FAST), _sc(spec.scenario)
    B, T = 120, 6
    ri, cand, wt, widx, ul = _batch(spec, B, seed=8)
    ris, w, tw, idx, ult = _dev(engine, ri, cand, wt, widx, ul)
    Bw = w.shape[1]
    assert Bw < B
    with torch.no_grad():
        plain = _ep(ris, w, idx, tw, ult, p, sc, T)
    rg, wg, tg = (x.clone().requires_grad_(True) for x in (ris, w, tw))
    ret = _ep(rg, wg, idx, tg, ult, p, sc, T)
    assert torch.equal(ret.detach(), plain)                  # the forward is untouched by autograd
    rb = torch.as_tensor(np.random.default_rng(1).normal(size=B), dtype=torch.float32, device=engine.device)
    g1 = torch.autograd.grad(ret, (rg, wg, tg), rb, retain_graph=True)
    g2 = torch.autograd.grad(ret, (rg, wg, tg), rb)
    assert all(torch.equal(a, b) for a, b in zip(g1, g2))     # deterministic, bit for bit
    fwd = engine.episodes_soa(p, sc, ris, w, Bw, tw, T, weight_idx=idx, unlucky_idx=ult, trace=True)
    ref = engine.episodes_vjp_soa(p, sc, w, Bw, tw, T, fwd["states"], fwd["best"], fwd["controls"], rb, idx)
    assert torch.equal(g1[0], ref["robot_init_bar"])
    per = ref["plan_weights_bar"].cpu().numpy().astype(np.float64)
    want = np.zeros((p.K, Bw))
    for b in range(B):
        want[:, widx[b]] += per[:, b]
    np.testing.assert_allclose(g1[1].cpu().numpy(), want, rtol=1e-5, atol=1e-5 * np.abs(want).max())
    tw_want = ref["true_weights_bar"].cpu().numpy().astype(np.float64).sum(axis=1)
    np.testing.assert_allclose(g1[2].cpu().numpy(), tw_want, rtol=1e-5, atol=1e-5 * np.abs(tw_want).max())
    # one weight vector for every world: its gradient is the batch sum
    w1 = w[:, :1].contiguous().requires_grad_(True)
    ret1 = _ep(ris, w1, None, tw, ult, p, sc, T)
    gw1, = torch.autograd.grad(ret1, (w1,), rb)
    fwd1 = engine.episodes_soa(p, sc, ris, w[:, :1].contiguous(), 1, tw, T, unlucky_idx=ult, trace=True)
    ref1 = engine.episodes_vjp_soa(p, sc, w[:, :1].contiguous(), 1, tw, T, fwd1["states"], fwd1["best"],
                                   fwd1["controls"], rb)
    np.testing.assert_allclose(gw1.cpu().numpy()[:, 0], ref1["plan_weights_bar"].cpu().numpy().astype(np.float64).sum(1),
                               rtol=1e-5, atol=1e-5 * ref1["plan_weights_bar"].abs().sum(1).max().item())


def test_gradient_step_changes_the_mean_return_as_predicted(engine):
    """A small step along the gradient of the mean return (every world with its own weight vector) changes it by what
    the gradient predicts, on finite_horizon worlds the oracle reproduces and whose return responds linearly over the
    step (no start switch inside it)."""
    spec = _spec("finite_horizon", 5, False)
    p, sc = _pp(spec.params, ocd.MATH_PRECISE), _sc(spec.scenario)
    B0, T = 96, 15
    ri, cand, wt, widx, _ = _batch(spec, B0, seed=21)
    wfull = cand[widx]
    _, spread = episode_conditioning(spec, ri, wfull, wt, T)
    keep = np.nonzero(spread < 1e-6)[0]
    dev = engine.device
    ris = torch.as_tensor(ri[keep].T.copy(), device=dev)
    w0 = torch.as_tensor(wfull[keep].T.copy(), device=dev)
    tw = torch.as_tensor(wt, device=dev)

    def mean_ret(w):
        return _ep(ris, w, None, tw, None, p, sc, T).mean()
    wg = w0.clone().requires_grad_(True)
    L0 = mean_ret(wg)
    g, = torch.autograd.grad(L0, wg)
    step = 1e-4 * g / g.norm(dim=0, keepdim=True)
    with torch.no_grad():
        r0 = _ep(ris, w0, None, tw, None, p, sc, T)
        d1 = _ep(ris, w0 + step, None, tw, None, p, sc, T) - r0
        d2 = _ep(ris, w0 + 0.5 * step, None, tw, None, p, sc, T) - r0
    lin = ((d1 - 2 * d2).abs() <= 0.02 * d1.abs()) & (d1.abs() > 0)
    assert lin.sum().item() >= 12, lin.sum().item()
    predicted = float((g * step)[:, lin].sum()) * len(keep)        # d mean / d w_b = grad of world b / n
    actual = float(d1[lin].sum())
    assert 0.9 <= actual / predicted <= 1.1, (actual, predicted)


# ---- MPC_ORD ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("scenario", ["finite_horizon", "replanning"])
def test_eval_weights_grad_objective_and_bookkeeping(engine, scenario):
    """eval_weights_grad's objective is eval_weights's bit for bit, and both advance history, iteration counter, the
    car's weights and initial state, the final world and the replanning reset toggle alike -- also when mixed."""
    from l4dc_mpc_ocd_b200.experiments import run_mpc_ord
    from l4dc_mpc_ocd_b200.interact_drive.reward_design.mpc_ord import MPC_ORD
    env = run_mpc_ord.envs[scenario]
    ms = []
    for _ in range(2):
        car, world, inits = env["make_env"](env_seeds=[1000000, 1000001, 1000002], debug=False)
        ms.append(MPC_ORD(world, car, inits, env["eval_horizon"], num_samples=env["num_eval_samples"], verbose=False))
    a, b = ms
    rng = np.random.default_rng(2)
    for i in range(3):
        w = a.designer_weights + 0.05 * rng.normal(size=a.weight_dim)
        oa = a.eval_weights(w)
        ob, g = b.eval_weights_grad(w) if i != 1 else (b.eval_weights(w), np.zeros(b.weight_dim))
        assert oa == ob, (i, oa, ob)
        assert g.shape == (a.weight_dim,) and np.isfinite(g).all()
        assert a.iter == b.iter and a.kernel_launches == b.kernel_launches
        assert [tuple(np.asarray(x).tolist()) for x, _ in a.history] == [tuple(np.asarray(x).tolist()) for x, _ in b.history]
        assert [v for _, v in a.history] == [v for _, v in b.history]
        assert np.array_equal(np.asarray(a.car.weights), np.asarray(b.car.weights))
        assert np.array_equal(np.asarray(a.car.init_state), np.asarray(b.car.init_state))
        for ca, cb in zip(a.world.cars, b.world.cars):
            assert np.array_equal(np.asarray(ca.state), np.asarray(cb.state))
        assert getattr(a.world, "unlucky_car_idx", None) == getattr(b.world, "unlucky_car_idx", None)
