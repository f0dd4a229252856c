"""L-BFGS episodes and ocd_episode_implicit_vjp_batch without a GPU: the workspace formula, the argument checks that run
before any CUDA call, the kernel form of L-BFGS episodes, the fake-tensor shapes of
torch.ops.ocd_b200.episodes_implicit_vjp and of episodes' backward under L-BFGS params, and MPC_ORD's planner option."""
import ctypes as C

import pytest
import torch

import l4dc_mpc_ocd_b200 as ocd

N = ocd._native


def _lbfgs(**kw):
    return ocd.PlannerParams(**{"H": 5, "n_iter": 10, "optimizer": ocd.OPT_LBFGS, **kw})


def _ws_bytes(p, T, B):
    n = C.c_size_t(123)
    rc = N.lib.ocd_episode_implicit_vjp_workspace_bytes(C.addressof(p), T, B, C.byref(n))
    return rc, n.value


def test_workspace_formula():
    for H, L, T, B in ((5, 3, 15, 256), (6, 3, 1, 1), (5, 2, 20, 4097), (16, 3, 3, 10)):
        lane_x = (-0.1, 0.0, 0.1) if L == 3 else (-0.05, 0.05)
        p = _lbfgs(H=H, lane_x=lane_x)
        rc, n = _ws_bytes(p.c_struct(), T, B)
        # Jacobian rows [T][2][K + 4][B], plans [T][H][2][B], status and held masks [T][B]; no iterate store
        assert rc == N.OK and n == (T * 2 * (p.K + 4) * B + T * H * 2 * B + 2 * T * B) * 4, (H, L, T, B)
    assert _ws_bytes(_lbfgs().c_struct(), 0, 64) == (N.OK, 0)
    assert _ws_bytes(_lbfgs().c_struct(), 15, 0) == (N.OK, 0)
    assert _ws_bytes(_lbfgs().c_struct(), 15, -1)[0] == N.EINVAL
    assert _ws_bytes(_lbfgs().c_struct(), -1, 8)[0] == N.EINVAL
    assert _ws_bytes(_lbfgs(H=17).c_struct(), 15, 8)[0] == N.EUNSUP
    # the SGD planner has the unrolled derivative
    assert _ws_bytes(ocd.PlannerParams().c_struct(), 15, 8)[0] == N.EUNSUP
    ps = _lbfgs().c_struct()
    assert N.lib.ocd_episode_implicit_vjp_workspace_bytes(C.addressof(ps), 15, 8, None) == N.EINVAL


def _sc(n_other=1, kind=0, plan_len=0):
    s = ocd.Scenario(init_state=[[0.0, -0.6, 0.5, 1.57]] * n_other, kind=[kind] * n_other, friction=[0.0] * n_other,
                     control=[[0.0, 0.0]] * n_other).c_struct()
    s.plan_len[0] = plan_len
    return s


def _ivjp(p, B, ws_bytes, T=2, sc=True, scs=None, states=True, best=True, controls=True, rbar=True, wbar=True,
          tw=True, w=True, Bw=1, ws=True):
    buf = (C.c_float * 512)()
    ib = (C.c_int32 * 64)()
    s = scs if scs is not None else _sc()
    return N.lib.ocd_episode_implicit_vjp_batch(C.addressof(p), C.addressof(s) if sc else None, buf if w else None, Bw,
                                                None, buf if tw else None, T, buf if states else None,
                                                ib if best else None, buf if controls else None,
                                                buf if rbar else None, buf if wbar else None, None, None,
                                                buf if ws else None, ws_bytes, B, None)


def test_argument_checks_need_no_device():
    p = _lbfgs()
    ps = p.c_struct()
    B, T = 4, 2
    need = (T * 2 * (p.K + 4) * B + T * p.H * 2 * B + 2 * T * B) * 4
    # the SGD planner: ocd_episode_vjp_batch differentiates it
    assert _ivjp(ocd.PlannerParams(H=5, n_iter=2).c_struct(), B, need) == N.EUNSUP
    # the L-BFGS horizon limit, and shapes out of range
    assert _ivjp(_lbfgs(H=17).c_struct(), B, 10 ** 6) == N.EUNSUP
    assert _ivjp(_lbfgs(C=1).c_struct(), B, need) == N.EINVAL
    # a workspace one byte short, or none at all
    assert _ivjp(ps, B, need - 1) == N.EINVAL
    assert _ivjp(ps, B, need, ws=False) == N.EINVAL
    assert _ivjp(ps, -1, need) == N.EINVAL
    assert _ivjp(ps, B, need, T=-1) == N.EINVAL
    assert _ivjp(ps, B, need, sc=False) == N.EINVAL
    assert _ivjp(ps, B, need, scs=_sc(n_other=2)) == N.EINVAL                # C = 2 has one other car
    assert _ivjp(ps, B, need, scs=_sc(kind=2)) == N.EINVAL
    assert _ivjp(ps, B, need, scs=_sc(kind=1, plan_len=N.MAX_PLAN + 1)) == N.EINVAL
    for missing in ("states", "best", "controls", "rbar", "wbar", "tw", "w"):
        assert _ivjp(ps, B, need, **{missing: False}) == N.EINVAL, missing
    assert _ivjp(ps, B, need, Bw=3) == N.EINVAL                # 3 weight vectors for 4 worlds without an index
    # nothing to do
    assert _ivjp(ps, 0, 0, states=False, best=False, controls=False, rbar=False, wbar=False, ws=False) == N.OK


def test_engine_has_no_cpu_fallback():
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    p = _lbfgs()
    need = (2 * 2 * (p.K + 4) * 4 + 2 * p.H * 2 * 4 + 2 * 2 * 4) * 4
    assert _ivjp(p.c_struct(), 4, need) == N.ECUDA
    # the forward is accepted up to the launch
    buf = (C.c_float * 256)()
    sc = _sc()
    ret = (C.c_float * 4)()
    assert N.lib.ocd_episode_batch(C.addressof(p.c_struct()), C.addressof(sc), buf, None, buf, 1, None, buf, None,
                                   0, 3, ret, None, None, None, None, 4, None) == N.ECUDA


def test_kernel_form_of_lbfgs_episodes():
    for B in (1, 45, 4096, 65536):
        assert ocd.kernel_form(_lbfgs(), B, episode=True) == "throughput"
        assert ocd.kernel_form(_lbfgs(H=16, extra_inits=True), B, episode=True) == "throughput"
    with pytest.raises(ValueError):
        ocd.kernel_form(_lbfgs(H=17), 45, episode=True)


def test_fake_shapes_and_backward():
    """Autograd through ocd_b200::episodes with L-BFGS params, traced with fake tensors: the backward runs the implicit
    op and the gradients have the shapes of robot_init, plan_weights and true_weights."""
    from torch._subclasses.fake_tensor import FakeTensorMode
    from l4dc_mpc_ocd_b200 import torch_ops as T_
    p = _lbfgs(C=3, lane_x=(-0.05, 0.05), other_mode=1, extra_inits=True)
    sc = ocd.Scenario(init_state=[[0.0, -0.7, 0.8, 1.57]] * 2, kind=[1, 1], friction=[0.2, 0.2],
                      control=[[0.0, 0.0]] * 2, plan=[[[0.0, 0.0], [0.7, 2.7]]] * 2, critical_t=4)
    B, T = 40, 6
    with FakeTensorMode():
        for Bw, idx in ((1, None), (7, torch.zeros(B, dtype=torch.int32, device="cpu"))):
            ri = torch.empty((4, B), device="cpu", requires_grad=True)
            w = torch.empty((p.K, Bw), device="cpu", requires_grad=True)
            tw = torch.empty((p.K,), device="cpu", requires_grad=True)
            ret = torch.ops.ocd_b200.episodes(ri, w, idx, tw, None, T_.pack_params(p), T_.pack_scenario(sc), T)
            gr, gw, gt = torch.autograd.grad((ret * ret).sum(), (ri, w, tw))
            assert gr.shape == (4, B) and gw.shape == (p.K, Bw) and gt.shape == (p.K,)
            _, ctl, best, states = torch.ops.ocd_b200.episodes_trace(ri, w, idx, tw, None, T_.pack_params(p),
                                                                     T_.pack_scenario(sc), T)
            pb, rb, tb = torch.ops.ocd_b200.episodes_implicit_vjp(w, idx, tw, states, best, ctl, ret,
                                                                  T_.pack_params(p), T_.pack_scenario(sc), T)
            assert pb.shape == (p.K, B) and rb.shape == (4, B) and tb.shape == (p.K, B)


def test_mpc_ord_planner_option():
    """planner_optimizer / planner_iters set the episode params; the default leaves the car's SGD planner alone."""
    from l4dc_mpc_ocd_b200.interact_drive.reward_design.mpc_ord import MPC_ORD, finite_horizon_env
    car, env, inits = finite_horizon_env(debug=False)
    base = MPC_ORD(env, car, inits, 5, verbose=False).program.params
    assert base.optimizer == ocd.OPT_SGD
    lb = MPC_ORD(env, car, inits, 5, verbose=False, planner_optimizer=ocd.OPT_LBFGS, planner_iters=40).program.params
    assert lb.optimizer == ocd.OPT_LBFGS and lb.n_iter == 40
    assert (lb.H, lb.C, tuple(lb.lane_x), lb.lr) == (base.H, base.C, tuple(base.lane_x), base.lr)
    assert MPC_ORD(env, car, inits, 5, verbose=False, planner_optimizer=ocd.OPT_LBFGS).program.params.n_iter == \
        base.n_iter
