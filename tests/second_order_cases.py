"""Inputs of the second-order comparisons (tests/test_gpu_second_order.py), shared with the CPU check of their reference
(tests/test_autodiff64_cpu.py).  No engine import: the reference's own tests do not need the native library."""
import numpy as np

import oracle as O

LANES = {1: (0.0,), 2: (-0.05, 0.05), 3: (-0.1, 0.0, 0.1), 4: (-0.15, -0.05, 0.05, 0.15)}


def params(H, C, L, other_mode, **kw) -> O.OracleParams:
    return O.OracleParams(H=H, C=C, lane_x=LANES[L], num_lanes=L, other_mode=other_mode,
                          target_speed=1.2 if L == 2 else 1.0, **kw)


def make_inputs(op: O.OracleParams, B: int, seed: int, Bo=None, controls: bool = True):
    """-> dict(world [B, C, 4], u [B, H, 2], w [B, K], oc [Bo, C-1, H, 2] or None) with every curvature term on."""
    rng = np.random.default_rng(seed)
    H, Cc, L = op.H, op.C, op.L
    ts = float(np.float32(op.target_speed))
    lo, thr = 0.05 * op.num_lanes - 0.05, 0.05 * op.num_lanes
    kind = np.arange(B) % 4
    x = np.where(kind == 0, rng.choice(LANES[L], B) + rng.uniform(-0.03, 0.03, B),
                 np.where(kind == 1, rng.uniform(lo, thr + 0.01, B),                # inside the fence ramp, +x side
                          np.where(kind == 2, -rng.uniform(lo, thr + 0.01, B),      # and the -x side
                                   rng.uniform(-thr - 0.05, thr + 0.05, B))))
    y = rng.uniform(-1.0, 0.0, B)
    th = np.pi / 2 + rng.uniform(-0.5, 0.5, B) * min(1.0, 8.0 / H)     # long rollouts: stay near the lanes
    fast = rng.random(B) < 0.3                                                       # over the speed bound
    v = np.where(fast, rng.uniform(3.6, 4.5, B) * ts, rng.uniform(0.2, 1.6, B))
    world = np.zeros((B, Cc, 4))
    world[:, 0] = np.stack([x, y, v, th], 1)
    for c in range(1, Cc):
        near = (c == 1) | (rng.random(B) < 0.5)                                      # car 1 always starts close by
        world[:, c, 0] = np.where(near, x + rng.uniform(-0.07, 0.07, B), rng.choice(LANES[L], B))
        world[:, c, 1] = np.where(near, y + rng.uniform(-0.1, 0.25, B), rng.uniform(-1.0, 1.0, B))
        world[:, c, 2] = np.where(near, np.minimum(v, 1.6) * rng.uniform(0.7, 1.1, B), rng.uniform(0.2, 1.2, B))
        world[:, c, 3] = np.pi / 2 + rng.uniform(-0.1, 0.1, B)
    u = rng.normal(size=(B, H, 2)) * np.array([1.0, 1.5])
    on_a, on_w = rng.random((B, H)) < 0.12, rng.random((B, H)) < 0.12               # on a limit and beyond
    u[..., 1] = np.where(on_w, rng.choice([4.0, -4.0, 4.4, -4.6], (B, H)), u[..., 1])
    spd = v.copy()
    for t in range(H):          # accelerations about the speed-holding one, so that long rollouts stay finite
        a = np.where(on_a[:, t], rng.choice([4.0, -8.0, 4.7, -8.6], B),
                     op.friction * spd ** 2 + 2.0 * (v - spd) + u[:, t, 0])
        u[:, t, 0] = a
        spd = spd + (np.clip(a, -8.0, 4.0) - op.friction * spd ** 2) * op.dt
    w = -rng.uniform(0.1, 1.0, (B, op.K)) * np.where(rng.random((B, op.K)) < 0.15, -1.0, 1.0)
    oc = None
    if op.other_mode == 1:
        oc = (0.3 * rng.normal(size=(Bo or B, Cc - 1, H, 2))).astype(np.float32)
    return dict(world=world.astype(np.float32), u=u.astype(np.float32) if controls else None,
                w=w.astype(np.float32), oc=oc)



# (H, C, L, other_mode, Bo, B): H in {1, 2, 5, 16, 64}, C in {2, 3, 5, 8}, L in {1, 2, 3, 4}, Bo == B and Bo == 1
FEATURE_SHAPES = [(1, 2, 1, 0, None, 96), (2, 3, 2, 1, "B", 96), (5, 2, 3, 0, None, 96), (5, 5, 4, 1, 1, 96),
                  (16, 8, 3, 0, None, 50), (64, 3, 2, 1, 1, 24), (64, 8, 4, 0, None, 50)]


def feature_case(H, C, L, other_mode, Bo, B):
    op = params(H, C, L, other_mode)
    inp = make_inputs(op, B, seed=1000 + 37 * H + 5 * C + L, Bo=B if Bo == "B" else Bo)
    return op, inp


# One shape per iteration code the reverse pass re-runs (ocd_api.cu's dispatch; the kernel named is the fast-math
# one, precise math runs OCD_DISPATCH's), with the budgets n_iter checked: (H, C, L, other_mode, extra, lr, B), n_iters.
# A long horizon takes a small lr: with a larger one the float64 plan itself runs away (negative speed) in 2-3 steps.
VJP_CASES = [
    ((5, 2, 3, 0, False, 0.1, 64), (0, 1, 2, 3)),       # <5, 1, 3>: register-resident, the finite_horizon shape
    ((5, 6, 3, 0, False, 0.1, 64), (0, 1, 2, 3)),       # <5, 5, 3>: compile-time car count (precise <5, 0, 3>)
    ((6, 4, 4, 1, True, 0.1, 64), (0, 1, 2, 3)),        # <0, 0, 0> with extra-init starts and known controls
    ((15, 2, 3, 0, False, 0.1, 160), (0, 1, 2)),        # <15, 1, 3>: the Q kernels (sgd_iteration_q)
    ((15, 3, 3, 0, False, 0.1, 128), (0, 1, 3)),        # <15, 2, 3>: constant-segment adjoint (OCD_IS_SEGC)
    ((12, 2, 3, 0, False, 0.1, 128), (0, 1, 3)),        # <0, 1, 3>: runtime horizon, one other car
    ((12, 3, 2, 1, False, 0.1, 128), (0, 1, 3)),        # <0, 0, 0>: runtime horizon, cars and lanes
    ((50, 2, 3, 0, False, 3e-4, 32), (0, 1, 2)),        # <50, 1, 3>: constant segments, linear other-car slab
    ((64, 8, 3, 0, True, 3e-4, 16), (0, 1, 2)),         # <0, 0, 3> at OCD_MAX_H and OCD_MAX_OTHER, extra inits
]
VJP_SHAPES = [s for s, _ in VJP_CASES]


def vjp_case(shape, n_iter):
    H, Cc, L, other_mode, extra, lr, B = shape
    op = params(H, Cc, L, other_mode, extra_inits=extra, lr=lr, n_iter=n_iter)
    inp = make_inputs(op, B, seed=2000 + 13 * H + Cc, controls=False)
    pbar = np.random.default_rng(H + Cc).normal(size=(B, H, 2)).astype(np.float32)
    return op, inp, pbar



IVJP_SHAPES = [(5, 2, 3, 0, None), (5, 3, 2, 1, "B"), (6, 4, 4, 1, 1), (16, 2, 3, 0, None)]
