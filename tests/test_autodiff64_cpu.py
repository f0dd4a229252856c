"""oracle/autodiff64.py pinned to the C oracle before any GPU comparison uses it: the reward and its gradient in
float64, the unrolled SGD iterates, the Hessian's symmetry and its agreement with differences of the oracle's gradient,
and the tie conventions of the lane-min and collision features.  CPU only."""
import numpy as np
import pytest
import torch

import oracle as O
from oracle.autodiff64 import Reference

from second_order_cases import FEATURE_SHAPES, IVJP_SHAPES, VJP_SHAPES, feature_case, make_inputs, params, vjp_case


def _all_shapes():
    """(op, inputs) of every shape the GPU comparisons use, with random weights and controls."""
    out = []
    for s in FEATURE_SHAPES:
        out.append((f"feature{s}",) + feature_case(*s))
    for s in VJP_SHAPES:
        op, inp, _ = vjp_case(s, 3)
        out.append((f"vjp{s}", op, inp))
    for H, Cc, L, om, Bo in IVJP_SHAPES:
        op = params(H, Cc, L, om, optimizer=1)
        out.append((f"ivjp{(H, Cc, L, om, Bo)}", op, make_inputs(op, 16, seed=H + Cc, Bo=Bo if Bo == 1 else None)))
    return out


SHAPES = _all_shapes()


def _oc(inp, b):
    oc = inp["oc"]
    return None if oc is None else oc[0 if oc.shape[0] == 1 else b].astype(np.float64)


@pytest.mark.parametrize("name,op,inp", SHAPES, ids=[s[0] for s in SHAPES])
def test_reward_and_gradient_equal_the_oracle(name, op, inp):
    n = min(len(inp["world"]), 12)
    rng = np.random.default_rng(op.H)
    u = inp["u"] if inp["u"] is not None else (rng.normal(size=(len(inp["world"]), op.H, 2)) * 1.5)
    r, g = Reference(op).batch_reward(inp["world"][:n], u[:n], inp["w"][:n],
                                      None if inp["oc"] is None else inp["oc"][:n] if inp["oc"].shape[0] > 1
                                      else inp["oc"])
    for b in range(n):
        R, G = O.mpc_reward(op, inp["world"][b].astype(np.float64), np.asarray(u[b], np.float64),
                            inp["w"][b].astype(np.float64), other_controls=_oc(inp, b), dtype=np.float64)
        assert abs(r[b] - R) <= 1e-12 * max(1.0, abs(R)), (b, r[b], R)
        G = np.asarray(G).reshape(-1)
        assert np.abs(g[b] - G).max() <= 1e-12 * max(1.0, np.abs(G).max()), b


@pytest.mark.parametrize("shape", [s for s in VJP_SHAPES if s[0] <= 12] + [(6, 3, 3, 1, True, 0.1, 6)])
@pytest.mark.parametrize("n_iter", [1, 3])
def test_sgd_iterates_equal_the_oracle(shape, n_iter):
    """sgd_plan of every start equals the oracle's f64 generate_plan (all_plans), extra-init starts included."""
    op, inp, _ = vjp_case(shape, n_iter)
    B = min(len(inp["world"]), 6)
    ref = Reference(op)
    for s in range(op.S):
        oc = None if inp["oc"] is None else inp["oc"][:B]
        plans = ref.batch_sgd_iterates(inp["world"][:B], inp["w"][:B], [s] * B, n_iter, oc)[:, -1]
        for b in range(B):
            r = O.generate_plan(op, inp["world"][b].astype(np.float64), inp["w"][b].astype(np.float64),
                                other_controls=_oc(inp, b), dtype=np.float64, all_plans=True)
            want = np.asarray(r["all_plans"][s]).reshape(-1)
            assert np.abs(plans[b] - want).max() <= 1e-12 * max(1.0, np.abs(want).max()), (s, b)


@pytest.mark.parametrize("shape", [(5, 3, 3, 0, None, 12), (8, 5, 2, 1, "B", 12), (16, 2, 4, 0, None, 8)])
def test_hessian_is_symmetric_and_matches_oracle_differences(shape):
    """hessian_u is symmetric; where central differences of the oracle's f64 gradient agree at two step sizes (no
    kink within the step), they agree with it."""
    op, inp = feature_case(*shape)
    ref = Reference(op)
    Hs = ref.batch_hessian_u(inp["world"], inp["u"], inp["w"], inp["oc"])
    assert np.array_equal(Hs, Hs.transpose(0, 2, 1)) or np.abs(Hs - Hs.transpose(0, 2, 1)).max() <= 1e-12 * \
        np.abs(Hs).max()
    n, compared = 2 * op.H, 0
    for b in range(len(inp["world"])):
        x, w, u = inp["world"][b].astype(np.float64), inp["w"][b].astype(np.float64), inp["u"][b].astype(np.float64)

        def fd(h):
            D = np.zeros((n, n))
            for i in range(n):
                e = np.zeros(n)
                e[i] = h
                gp = O.mpc_reward(op, x, (u.reshape(-1) + e).reshape(op.H, 2), w, _oc(inp, b), np.float64)[1]
                gm = O.mpc_reward(op, x, (u.reshape(-1) - e).reshape(op.H, 2), w, _oc(inp, b), np.float64)[1]
                D[:, i] = (np.asarray(gp) - np.asarray(gm)).reshape(-1) / (2 * h)
            return D
        d1, d2 = fd(1e-5), fd(5e-6)
        scale = max(1.0, np.abs(Hs[b]).max())
        agree = np.abs(d1 - d2).max(axis=0) <= 1e-5 * scale          # per column: no kink along that control
        assert np.abs(Hs[b][:, agree] - d2[:, agree]).max(initial=0.0) <= 1e-5 * scale, b
        compared += agree.sum()
    assert compared >= 0.8 * n * len(inp["world"]), compared


def test_first_minimum_and_first_maximum_win():
    """Exact ties: the lane-min feature takes the first lane's derivative and the collision feature the first car's,
    not the split torch.amin / amax would give."""
    op = params(1, 3, 2, 0)
    ref = Reference(op)
    s = torch.tensor([0.0, 0.0, 1.0, np.pi / 2], dtype=torch.float64)        # halfway between the lanes +-0.05
    others = torch.tensor([[0.02, 0.05, 0.5, np.pi / 2], [0.02, 0.05, 0.5, np.pi / 2]], dtype=torch.float64)
    J = torch.func.jacrev(ref.features)(s, others)
    L = op.L
    assert torch.equal(J[1 + L, 0], J[1, 0]) and J[1, 0] != J[2, 0]
    Jo = torch.func.jacrev(ref.features, argnums=1)(s, others)[2 + L]
    assert torch.all(Jo[0, :2] != 0) and torch.all(Jo[1] == 0)


def test_branch_margin_counts_the_clip_limits_of_computed_controls_only():
    op = params(2, 2, 3, 0)
    ref = Reference(op)
    world = torch.tensor([[0.0, -0.5, 1.0, np.pi / 2], [0.0, 5.0, 1.0, np.pi / 2]], dtype=torch.float64)
    u = torch.tensor([4.0 - 1e-7, -3.0, -7.0, 0.3], dtype=torch.float64)
    oc = torch.zeros(1, 2, 2, dtype=torch.float64)
    assert float(ref.branch_margin(u, world, oc)) > 1e-3
    assert float(ref.branch_margin(u, world, oc, computed=True)) == pytest.approx(1e-7, rel=1e-6)
