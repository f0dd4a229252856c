"""ocd_solve_implicit_vjp_batch without a GPU: the argument checks that run before any CUDA call, and the fake-tensor
shapes of torch.ops.ocd_b200.solve_implicit_vjp and of solve's backward with L-BFGS params."""
import ctypes as C

import pytest
import torch

import l4dc_mpc_ocd_b200 as ocd

N = ocd._native


def _ivjp(p, B, world=True, plan=True, plan_bar=True, wbar=True, Bw=1, idx=None, weights=True, oc=None, Bo=0):
    buf = (C.c_float * 256)()
    return N.lib.ocd_solve_implicit_vjp_batch(C.addressof(p), buf if world else None, oc, Bo,
                                              buf if weights else None, Bw, idx, buf if plan else None,
                                              buf if plan_bar else None, buf if wbar else None, None, None, B, None)


def _lbfgs(**kw):
    return ocd.PlannerParams(**{"H": 5, "n_iter": 10, "optimizer": ocd.OPT_LBFGS, **kw}).c_struct()


def test_argument_checks_need_no_device():
    ps = _lbfgs()
    # the SGD plan has its own, exact, unrolled derivative
    assert _ivjp(ocd.PlannerParams(H=5, n_iter=10).c_struct(), 4) == N.EUNSUP
    # the L-BFGS horizon limit, and shapes out of range
    assert _ivjp(_lbfgs(H=17), 4) == N.EUNSUP
    assert _ivjp(ocd.PlannerParams(H=65, optimizer=ocd.OPT_LBFGS).c_struct(), 4) == N.EUNSUP
    assert _ivjp(_lbfgs(C=9), 4) == N.EUNSUP
    assert _ivjp(_lbfgs(C=1), 4) == N.EINVAL
    # missing arrays
    assert _ivjp(ps, 4, world=False) == N.EINVAL
    assert _ivjp(ps, 4, plan=False) == N.EINVAL
    assert _ivjp(ps, 4, plan_bar=False) == N.EINVAL
    assert _ivjp(ps, 4, wbar=False) == N.EINVAL
    assert _ivjp(ps, 4, weights=False) == N.EINVAL
    assert _ivjp(ps, -1) == N.EINVAL
    # weight tables: 3 vectors for 4 problems need an index; an empty table is refused
    assert _ivjp(ps, 4, Bw=3) == N.EINVAL
    assert _ivjp(ps, 4, Bw=0, idx=(C.c_int32 * 4)()) == N.EINVAL
    # known controls of the other cars: missing, or a Bo that is neither 1 nor B
    om = _lbfgs(other_mode=1)
    assert _ivjp(om, 4) == N.EINVAL
    assert _ivjp(om, 4, oc=(C.c_float * 64)(), Bo=3) == N.EINVAL
    # nothing to do
    assert _ivjp(ps, 0, world=False, plan=False, plan_bar=False, wbar=False, weights=False) == N.OK


def test_the_solve_vjp_still_refuses_lbfgs():
    lb = _lbfgs()
    n = C.c_size_t(0)
    assert N.lib.ocd_solve_vjp_workspace_bytes(C.addressof(lb), 4, C.byref(n)) == N.EUNSUP


def test_engine_has_no_cpu_fallback_for_the_implicit_vjp():
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    assert _ivjp(_lbfgs(), 4) == N.ECUDA


def test_fake_shapes():
    """The op and solve's backward under L-BFGS params, traced with fake tensors: the gradients have the shapes of
    world and weights, for a shared table (Bw = 1) and an indexed one (Bw < B)."""
    from torch._subclasses.fake_tensor import FakeTensorMode
    from l4dc_mpc_ocd_b200 import torch_ops as T
    p = ocd.PlannerParams(H=6, C=3, extra_inits=True, optimizer=ocd.OPT_LBFGS)
    B = 40
    with FakeTensorMode():
        for Bw, idx in ((1, None), (7, torch.zeros(B, dtype=torch.int32, device="cpu"))):
            world = torch.empty((p.C, 4, B), device="cpu", requires_grad=True)
            w = torch.empty((p.K, Bw), device="cpu", requires_grad=True)
            plan, losses, best = torch.ops.ocd_b200.solve(world, w, idx, None, T.pack_params(p))
            assert plan.shape == (p.H, 2, B)
            gw, gx = torch.autograd.grad((plan * plan).sum(), (w, world))
            assert gw.shape == (p.K, Bw) and gx.shape == (p.C, 4, B)
            wb, xb = torch.ops.ocd_b200.solve_implicit_vjp(world, w, idx, None, plan, plan, T.pack_params(p))
            assert wb.shape == (p.K, B) and xb.shape == (p.C, 4, B)
