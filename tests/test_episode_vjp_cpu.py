"""ocd_episode_vjp_batch without a GPU: the workspace sizes, the argument checks that run before any CUDA call, the
autograd wiring of torch.ops.ocd_b200.episodes traced with fake tensors, and the normalisation chain of
MPC_ORD.eval_weights_grad."""
import ctypes as C

import numpy as np
import pytest
import torch

import l4dc_mpc_ocd_b200 as ocd

N = ocd._native


def _ws_bytes(p, T, B):
    lo, full = C.c_size_t(123), C.c_size_t(456)
    rc = N.lib.ocd_episode_vjp_workspace_bytes(C.addressof(p), T, B, C.byref(lo), C.byref(full))
    return rc, lo.value, full.value


def test_workspace_sizes():
    for H, L, n_iter, T, B in ((5, 3, 100, 15, 256), (6, 3, 200, 1, 1), (5, 2, 100, 20, 4097), (15, 3, 0, 3, 10)):
        lane_x = (-0.1, 0.0, 0.1) if L == 3 else (-0.05, 0.05)
        p = ocd.PlannerParams(H=H, n_iter=n_iter, lane_x=lane_x)
        rc, lo, full = _ws_bytes(p.c_struct(), T, B)
        jac = T * 2 * (p.K + 4) * B * 4
        step = (n_iter + 1) * H * 2 * B * 4
        assert rc == N.OK and lo == jac + step and full == jac + T * step
    assert _ws_bytes(ocd.PlannerParams().c_struct(), 0, 64)[1:] == (0, 0)
    assert _ws_bytes(ocd.PlannerParams().c_struct(), 15, 0)[1:] == (0, 0)
    assert _ws_bytes(ocd.PlannerParams().c_struct(), 15, -1)[0] == N.EINVAL
    assert _ws_bytes(ocd.PlannerParams().c_struct(), -1, 8)[0] == N.EINVAL
    assert _ws_bytes(ocd.PlannerParams(H=65).c_struct(), 15, 8)[0] == N.EUNSUP
    assert _ws_bytes(ocd.PlannerParams(H=5, optimizer=ocd.OPT_LBFGS).c_struct(), 15, 8)[0] == N.EUNSUP
    lo, ps = C.c_size_t(0), ocd.PlannerParams().c_struct()
    assert N.lib.ocd_episode_vjp_workspace_bytes(C.addressof(ps), 15, 8, C.byref(lo), None) == N.EINVAL


def _sc(n_other=1, kind=0, plan_len=0):
    s = ocd.Scenario(init_state=[[0.0, -0.6, 0.5, 1.57]] * n_other, kind=[kind] * n_other, friction=[0.0] * n_other,
                     control=[[0.0, 0.0]] * n_other).c_struct()
    s.plan_len[0] = plan_len
    return s


def _vjp(p, B, ws_bytes, T=2, sc=True, scs=None, states=True, best=True, controls=True, rbar=True, wbar=True,
         tw=True, w=True, Bw=1, ws=True):
    buf = (C.c_float * 256)()
    ib = (C.c_int32 * 64)()
    s = scs if scs is not None else _sc()
    return N.lib.ocd_episode_vjp_batch(C.addressof(p), C.addressof(s) if sc else None, buf if w else None, Bw, None,
                                       buf if tw else None, T, buf if states else None, ib if best else None,
                                       buf if controls else None, buf if rbar else None, buf if wbar else None, None,
                                       None, buf if ws else None, ws_bytes, B, None)


def test_argument_checks_need_no_device():
    p = ocd.PlannerParams(H=5, n_iter=2)
    ps = p.c_struct()
    B, T = 4, 2
    need = T * 2 * (p.K + 4) * B * 4 + 3 * 5 * 2 * B * 4
    # L-BFGS plans are not differentiable through their line search
    assert _vjp(ocd.PlannerParams(H=5, n_iter=2, optimizer=ocd.OPT_LBFGS).c_struct(), B, need) == N.EUNSUP
    # a workspace one byte short, or none at all
    assert _vjp(ps, B, need - 1) == N.EINVAL
    assert _vjp(ps, B, need, ws=False) == N.EINVAL
    # bad shapes, scenarios and missing arrays
    assert _vjp(ocd.PlannerParams(H=65).c_struct(), B, 10 ** 6) == N.EUNSUP
    assert _vjp(ocd.PlannerParams(C=1).c_struct(), B, need) == N.EINVAL
    assert _vjp(ps, -1, need) == N.EINVAL
    assert _vjp(ps, B, need, T=-1) == N.EINVAL
    assert _vjp(ps, B, need, sc=False) == N.EINVAL
    assert _vjp(ps, B, need, scs=_sc(n_other=2)) == N.EINVAL                 # C = 2 has one other car
    assert _vjp(ps, B, need, scs=_sc(kind=2)) == N.EINVAL
    assert _vjp(ps, B, need, scs=_sc(kind=1, plan_len=N.MAX_PLAN + 1)) == N.EINVAL
    assert _vjp(ps, B, need, scs=_sc(kind=1, plan_len=-1)) == N.EINVAL
    for missing in ("states", "best", "controls", "rbar", "wbar", "tw", "w"):
        assert _vjp(ps, B, need, **{missing: False}) == N.EINVAL, missing
    assert _vjp(ps, B, need, Bw=3) == N.EINVAL                # 3 weight vectors for 4 worlds without an index
    # nothing to do
    assert _vjp(ps, 0, 0, states=False, best=False, controls=False, rbar=False, wbar=False, ws=False) == N.OK


def test_engine_has_no_cpu_fallback_for_the_episode_vjp():
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    p = ocd.PlannerParams(n_iter=2)
    need = 2 * 2 * (p.K + 4) * 4 * 4 + 3 * 5 * 2 * 4 * 4
    assert _vjp(p.c_struct(), 4, need) == N.ECUDA
    # T = 0 needs no trace, but its zeros are still written by a kernel
    assert _vjp(p.c_struct(), 4, 0, T=0, states=False, best=False, controls=False, ws=False) == N.ECUDA
    with pytest.raises(N.OcdCudaError):
        ocd.Engine(0)


def test_fake_shapes_and_backward():
    """Autograd through ocd_b200::episodes traced with fake tensors: the gradients have the shapes of robot_init,
    plan_weights and true_weights for a shared table (Bw = 1) and an indexed one; episodes_vjp and episodes_trace have
    the documented shapes."""
    from torch._subclasses.fake_tensor import FakeTensorMode
    from l4dc_mpc_ocd_b200 import torch_ops as T_
    p = ocd.PlannerParams(H=5, C=3, lane_x=(-0.05, 0.05), other_mode=1)
    sc = ocd.Scenario(init_state=[[0.0, -0.7, 0.8, 1.57]] * 2, kind=[1, 1], friction=[0.2, 0.2],
                      control=[[0.0, 0.0]] * 2, plan=[[[0.0, 0.0], [0.7, 2.7]]] * 2, critical_t=4)
    B, T = 40, 6
    with FakeTensorMode():
        for Bw, idx in ((1, None), (7, torch.zeros(B, dtype=torch.int32, device="cpu"))):
            ri = torch.empty((4, B), device="cpu", requires_grad=True)
            w = torch.empty((p.K, Bw), device="cpu", requires_grad=True)
            tw = torch.empty((p.K,), device="cpu", requires_grad=True)
            ret = torch.ops.ocd_b200.episodes(ri, w, idx, tw, None, T_.pack_params(p), T_.pack_scenario(sc), T)
            assert ret.shape == (B,)
            gr, gw, gt = torch.autograd.grad((ret * ret).sum(), (ri, w, tw))
            assert gr.shape == (4, B) and gw.shape == (p.K, Bw) and gt.shape == (p.K,)
            r2, ctl, best, states = torch.ops.ocd_b200.episodes_trace(ri, w, idx, tw, None, T_.pack_params(p),
                                                                      T_.pack_scenario(sc), T)
            assert r2.shape == (B,) and ctl.shape == (T, 2, B) and best.shape == (T, B) and best.dtype == torch.int32
            assert states.shape == (T, p.C, 4, B)
            pb, rb, tb = torch.ops.ocd_b200.episodes_vjp(w, idx, tw, states, best, ctl, ret, T_.pack_params(p),
                                                         T_.pack_scenario(sc), T)
            assert pb.shape == (p.K, B) and rb.shape == (4, B) and tb.shape == (p.K, B)


def test_normalisation_chain_matches_differences():
    """_planning_weights_vjp against central differences of the float64 normalisation chain, and of _planning_weights
    itself (float32 output, so a coarser step and tolerance)."""
    from l4dc_mpc_ocd_b200.interact_drive.reward_design.mpc_ord import MPC_ORD, _planning_weights_vjp
    rng = np.random.default_rng(4)

    def chain64(x):
        for _ in range(3):
            x = x / np.linalg.norm(x)
        return x
    for K, scale in ((7, 1.0), (6, 30.0), (7, 0.01)):
        w = rng.normal(size=K) * scale
        g = rng.normal(size=K)
        got = _planning_weights_vjp(w, g)
        for _ in range(3):
            d = rng.normal(size=K)
            h = 1e-6 * np.linalg.norm(w)
            want = g.dot(chain64(w + h * d) - chain64(w - h * d)) / (2 * h)
            assert abs(got.dot(d) - want) <= 1e-7 * max(1.0, abs(want)) / min(1.0, np.linalg.norm(w)), (got.dot(d), want)
            h = 1e-2 * np.linalg.norm(w)
            want32 = g.dot(MPC_ORD._planning_weights(w + h * d).astype(np.float64)
                           - MPC_ORD._planning_weights(w - h * d).astype(np.float64)) / (2 * h)
            assert abs(got.dot(d) - want32) <= 2e-3 * max(1.0, abs(want32)) / min(1.0, np.linalg.norm(w))
        # the normalisation is scale-invariant: the gradient is orthogonal to w
        assert abs(got.dot(w)) <= 1e-12 * np.linalg.norm(got) * np.linalg.norm(w) * 10
