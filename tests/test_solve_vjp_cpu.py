"""ocd_solve_vjp_batch without a GPU: the workspace size, the argument checks that run before any CUDA call, and the
autograd wiring of torch.ops.ocd_b200.solve traced with fake tensors."""
import ctypes as C

import pytest
import torch

import l4dc_mpc_ocd_b200 as ocd

N = ocd._native


def _ws_bytes(p, B):
    n = C.c_size_t(123)
    rc = N.lib.ocd_solve_vjp_workspace_bytes(C.addressof(p), B, C.byref(n))
    return rc, n.value


def test_workspace_size():
    for H, n_iter, B in ((5, 100, 256), (6, 200, 1), (64, 3, 4097), (15, 0, 10)):
        rc, n = _ws_bytes(ocd.PlannerParams(H=H, n_iter=n_iter).c_struct(), B)
        assert rc == N.OK and n == n_iter * H * 2 * B * 4
    assert _ws_bytes(ocd.PlannerParams().c_struct(), 0) == (N.OK, 0)
    assert _ws_bytes(ocd.PlannerParams().c_struct(), -1)[0] == N.EINVAL
    assert _ws_bytes(ocd.PlannerParams(H=65).c_struct(), 8)[0] == N.EUNSUP
    assert N.lib.ocd_solve_vjp_workspace_bytes(C.addressof(ocd.PlannerParams().c_struct()), 8, None) == N.EINVAL


def _vjp(p, B, ws_bytes, world=True, best=True, plan_bar=True, wbar=True, Bw=1, oc=None, Bo=0, ws=True):
    buf = (C.c_float * 64)()
    ib = (C.c_int32 * 64)()
    return N.lib.ocd_solve_vjp_batch(C.addressof(p), buf if world else None, oc, Bo, buf, Bw, None, None,
                                     ib if best else None, buf if plan_bar else None, buf if wbar else None, None,
                                     buf if ws else None, ws_bytes, B, None)


def test_argument_checks_need_no_device():
    p = ocd.PlannerParams(H=5, n_iter=2)
    ps = p.c_struct()
    need = 2 * 5 * 2 * 4 * 4
    # L-BFGS plans are not differentiable through their line search
    lb = ocd.PlannerParams(H=5, n_iter=2, optimizer=ocd.OPT_LBFGS).c_struct()
    assert _vjp(lb, 4, need) == N.EUNSUP
    assert _ws_bytes(lb, 4)[0] == N.EUNSUP
    # a workspace one byte short, or none at all
    assert _vjp(ps, 4, need - 1) == N.EINVAL
    assert _vjp(ps, 4, need, ws=False) == N.EINVAL
    # bad shapes and missing arrays
    assert _vjp(ocd.PlannerParams(H=65).c_struct(), 4, 10 ** 6) == N.EUNSUP
    assert _vjp(ocd.PlannerParams(C=1).c_struct(), 4, need) == N.EINVAL
    assert _vjp(ps, -1, need) == N.EINVAL
    assert _vjp(ps, 4, need, world=False) == N.EINVAL
    assert _vjp(ps, 4, need, best=False) == N.EINVAL
    assert _vjp(ps, 4, need, plan_bar=False) == N.EINVAL
    assert _vjp(ps, 4, need, wbar=False) == N.EINVAL
    assert _vjp(ps, 4, need, Bw=3) == N.EINVAL               # 3 weight vectors for 4 problems without an index
    assert _vjp(ocd.PlannerParams(other_mode=1, n_iter=2).c_struct(), 4, need) == N.EINVAL   # known controls missing
    # nothing to do
    assert _vjp(ps, 0, 0, world=False, best=False, plan_bar=False, wbar=False, ws=False) == N.OK


def test_engine_has_no_cpu_fallback_for_the_vjp():
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    p = ocd.PlannerParams(n_iter=2).c_struct()
    assert _vjp(p, 4, 2 * 5 * 2 * 4 * 4) == N.ECUDA


def test_fake_backward_shapes():
    """Autograd through ocd_b200::solve traced with fake tensors: the gradients have the shapes of world and weights,
    for a shared table (Bw = 1) and an indexed one (Bw < B)."""
    from torch._subclasses.fake_tensor import FakeTensorMode
    from l4dc_mpc_ocd_b200 import torch_ops as T
    p = ocd.PlannerParams(H=6, C=3, extra_inits=True)
    B = 40
    with FakeTensorMode():
        for Bw, idx in ((1, None), (7, torch.zeros(B, dtype=torch.int32, device="cpu"))):
            world = torch.empty((p.C, 4, B), device="cpu", requires_grad=True)
            w = torch.empty((p.K, Bw), device="cpu", requires_grad=True)
            plan, losses, best = torch.ops.ocd_b200.solve(world, w, idx, None, T.pack_params(p))
            assert plan.shape == (p.H, 2, B) and losses.shape == (p.S, B) and best.shape == (B,)
            gw, gx = torch.autograd.grad((plan * plan).sum(), (w, world))
            assert gw.shape == (p.K, Bw) and gx.shape == (p.C, 4, B)
            wb, xb = torch.ops.ocd_b200.solve_vjp(world, w, idx, None, best, plan, T.pack_params(p))
            assert wb.shape == (p.K, B) and xb.shape == (p.C, 4, B)
