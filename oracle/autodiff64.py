"""Exact second derivatives of the planner's reward by automatic differentiation.  TEST INFRASTRUCTURE ONLY (see
oracle/__init__.py).

`Reference` restates NaivePlanner.mpc_reward (interact_drive/planner/naive_planner.py:32-79) as a pure function of
torch tensors, op for op like torch_serial.py and the C oracle, and lets ``torch.func`` differentiate it to any
order.  There is no differencing step, so there is no truncation error and no kink to skip: the derivatives are
those of the selected branch, exactly, in the chosen dtype.  float64 is the reference; float32 measures what float32
rounding alone loses on a problem.

Conventions are the kernels' (and TensorFlow's gradients'), not torch's defaults:
- clip_by_value passes the derivative on the closed box: a control exactly on a limit is differentiable;
- tf.minimum(e2, bound) passes to e2 where e2 <= bound;
- the first of tied minima (lane features) and maxima (collision products) wins: ``argmin`` / ``argmax`` + gather,
  never ``amin`` / ``amax``, which split ties;
- where() routes nothing to the branch it did not select; |x| has derivative +1 at 0 (the kernels' ``x < 0 ? -x : x``);
- the constants are cast as the C oracle casts them: target_speed through float32, dt**2 and the threshold's
  ``threshold - width`` computed in double and cast once.

One problem: controls u [2H] (flat index 2t + c, as the ABI), world [C][4] (row 0 the planning car), weights [K],
other controls [C-1][H][2] (ignored unless other_mode == 1).  The batch methods take numpy arrays with a leading
batch axis, ``vmap`` the one-problem functions over it and return numpy arrays in the reference's dtype."""
from __future__ import annotations

import numpy as np
import torch
from torch.func import grad, hessian, jacfwd, jacrev, vjp, vmap

from .oracle import OracleParams

CLIP_A = (-8.0, 4.0)        # simulation_utils.py:13-14: max(min(acc, 4), -2 * 4)
CLIP_W = (-4.0, 4.0)
BUMP_HX, BUMP_HY = 0.08, 0.15
TURN = 5 * 0.13             # naive_planner.py:107-118: the starts' steering


class Reference:
    def __init__(self, p: OracleParams, dtype=torch.float64, chunk: int = 64):
        self.p, self.dtype, self.chunk = p, dtype, chunk
        self.H, self.C, self.L, self.K = p.H, p.C, p.L, p.K
        c = self._c
        self.dt, self.dt2, self.mu, self.lr = c(p.dt), c(p.dt * p.dt), c(p.friction), c(p.lr)
        ts = float(np.float32(p.target_speed))                         # np.float32(target_speed), merging.py:49
        self.ts, self.bound = c(ts), c(4.0 * ts * ts)
        self.lane_x = c(list(p.lane_x))
        thr, width = 0.05 * p.num_lanes, 0.05                          # merging.py:80-81
        self.thr_shape, self.thr_lo, self.thr_w = c(5.0 / width), c(thr - width), c(width)
        self.hx, self.hy = c(BUMP_HX), c(BUMP_HY)
        self.turn = c(TURN)
        self.half = c(0.5)      # a Python float factor would promote forward-mode tangents of 0-d tensors to float64

    def _c(self, x) -> torch.Tensor:
        return torch.tensor(x, dtype=self.dtype)

    # ---- the reward -------------------------------------------------------------------------------------------------
    def _f(self, q):
        qc = torch.where(q > 0, q, torch.full_like(q, 0.01))
        return torch.where(q > 0, torch.exp(-1 / (self.thr_shape * qc)), torch.zeros_like(q))

    def _threshold(self, z):
        q = z - self.thr_lo
        F1, F2 = self._f(q), self._f(self.thr_w - q)
        return F1 / (F1 + F2)

    @staticmethod
    def _bump(z, start, end):
        width, center = (end - start) / 2, (start + end) / 2
        n = (z - center) / width
        cond = n * n < 1
        nc = torch.where(cond, n, torch.zeros_like(n))
        return torch.where(cond, torch.exp(-1 / (1 - nc * nc) + 1), torch.zeros_like(n))

    def features(self, s, others):
        """s [4] the planning car, others [C-1][4] -> phi [K] (merging.py:51-83)."""
        x, y, v, th = s[0], s[1], s[2], s[3]
        e = v * torch.sin(th) - self.ts
        e2 = e * e
        speed = torch.where(e2 <= self.bound, e2, self.bound)
        lanes = ((x - self.lane_x) * -1) ** 2 * 10
        fmin = lanes.gather(0, torch.argmin(lanes).reshape(1))[0]
        ox, oy = others[:, 0], others[:, 1]
        prods = self._bump(x, ox - self.hx, ox + self.hx) * self._bump(y, oy - self.hy, oy + self.hy)
        best = prods.gather(0, torch.argmax(prods).reshape(1))[0]
        ax = torch.where(x < 0, -x, x)
        fence = (self._threshold(x) + self._threshold(-x)) * ax
        return torch.cat([speed.reshape(1), lanes, torch.stack([fmin, best, fence])])

    def _robot_step(self, s, a, om):
        a = torch.where(a > CLIP_A[1], self._c(CLIP_A[1]), torch.where(a < CLIP_A[0], self._c(CLIP_A[0]), a))
        om = torch.where(om > CLIP_W[1], self._c(CLIP_W[1]), torch.where(om < CLIP_W[0], self._c(CLIP_W[0]), om))
        x, y, v, th = s[0], s[1], s[2], s[3]
        total = a - self.mu * (v * v)
        dist = v * self.dt + (self.half * total) * self.dt2
        return torch.stack([x + torch.cos(th) * dist, y + torch.sin(th) * dist, v + total * self.dt,
                            th + om * self.dt])

    def _others_step(self, o, oc_t):
        """naive_planner.py:53-66: known controls (no friction, no clip) or constant velocity."""
        x, y, v, th = o[:, 0], o[:, 1], o[:, 2], o[:, 3]
        if self.p.other_mode == 1:
            a, om = oc_t[:, 0], oc_t[:, 1]
            dist = v * self.dt + (self.half * a) * self.dt2
            return torch.stack([x + torch.cos(th) * dist, y + torch.sin(th) * dist, v + a * self.dt,
                                th + om * self.dt], dim=1)
        return torch.stack([x + (torch.cos(th) * v) * self.dt, y + (torch.sin(th) * v) * self.dt, v, th], dim=1)

    def rollout(self, u, world, oc):
        """-> the planning car's states [H + 1][4] and the other cars' [H + 1][C-1][4]."""
        s, o = world[0], world[1:]
        S, O = [s], [o]
        for t in range(self.H):
            s, o = self._robot_step(s, u[2 * t], u[2 * t + 1]), self._others_step(o, oc[:, t])
            S.append(s)
            O.append(o)
        return torch.stack(S), torch.stack(O)

    def phi_sum(self, u, world, oc):
        """sum_t phi(s_{t+1}) [K]: the horizon-summed features (ocd_feature_jacobian_batch's phi_sum)."""
        S, O = self.rollout(u, world, oc)
        return sum(self.features(S[t], O[t]) for t in range(1, self.H + 1))

    def reward(self, u, world, w, oc):
        return (w * self.phi_sum(u, world, oc)).sum()

    def grad_u(self, u, world, w, oc):
        return grad(self.reward)(u, world, w, oc)

    def hessian_u(self, u, world, w, oc):
        return hessian(self.reward)(u, world, w, oc)

    def feature_jacobian(self, u, world, oc):
        """[K][2H]: row k is grad_u with the one-hot weights e_k."""
        return jacrev(self.phi_sum)(u, world, oc)

    def feature_hessian(self, u, world, oc):
        """[K][2H][2H]: hessian_u with the one-hot weights e_k."""
        return jacfwd(jacrev(self.phi_sum))(u, world, oc)

    def grad_u_mixed(self, u, world, w, oc):
        """d grad_u / d w [2H][K] and d grad_u / d world [2H][C][4]."""
        return jacfwd(self.grad_u, argnums=(2, 1))(u, world, w, oc)

    # ---- the fixed-budget SGD of one start (naive_planner.py:107-164) ------------------------------------------------
    def start(self, world, s):
        """The start s [2H] (0..2, or 3..5 with extra_inits: a0 = friction v0^2 from the robot's own speed)."""
        a0 = torch.where(s >= 3, self.mu * (world[0, 2] * world[0, 2]), self._c(0.0))
        r = s % 3
        om0 = torch.where(r == 1, -self.turn, torch.where(r == 2, self.turn, self._c(0.0)))
        return torch.stack([a0, om0]).repeat(self.H)

    def sgd_iterates(self, world, w, oc, s, n_iter: int):
        """u^0 .. u^N [N + 1][2H] with u^{n+1} = u^n - lr d(-R)/du (Keras SGD, momentum 0)."""
        u = self.start(world, s)
        its = [u]
        for _ in range(n_iter):
            u = u - self.lr * (-self.grad_u(u, world, w, oc))
            its.append(u)
        return torch.stack(its)

    def sgd_plan(self, world, w, oc, s, n_iter: int):
        return self.sgd_iterates(world, w, oc, s, n_iter)[-1]

    def sgd_vjp(self, world, w, oc, s, n_iter: int, plan_bar):
        """plan_bar . d plan / d (w, world) -> (weights_bar [K], world_bar [C][4])."""
        _, pull = vjp(lambda w_, x_: self.sgd_plan(x_, w_, oc, s, n_iter), w, world)
        return pull(plan_bar)

    def sgd_vjp_along(self, world, w, oc, s, its, plan_bar):
        """sgd_vjp with the iterates' values taken from its [N][2H] (another run's u^0 .. u^{N-1}, e.g. the GPU's
        fast-math forward) and only their derivatives from this run: the exact reverse pass along that trajectory."""
        n_iter = its.shape[0]

        def plan(w_, x_):
            u = self.start(x_, s)
            for n in range(n_iter):
                u = its[n] + (u - u.detach())
                u = u - self.lr * (-self.grad_u(u, x_, w_, oc))
            return u
        _, pull = vjp(plan, w, world)
        return pull(plan_bar)

    # ---- where a branch decision could go the other way ---------------------------------------------------------------
    def branch_margin(self, u, world, oc, computed: bool = False):
        """The smallest distance of any branch decision along the rollout of u to its threshold: the speed feature's
        bound, the gap between the two smallest lane features, 1 - n^2 of every bump, the relative gap between the
        two largest bump products (where one is nonzero), the fence's q and width - q on both sides, |x| for abs
        (where the fence's ramp factor is nonzero), and with `computed` the clip limits of the controls.  Controls
        given as inputs are the same numbers in every precision, so their clip decisions cannot differ: only controls
        the planner computes (the SGD iterates) count."""
        inf = self._c(float("inf"))
        m = []
        if computed:
            a, om = u[0::2], u[1::2]
            m += [torch.abs(a - CLIP_A[0]), torch.abs(a - CLIP_A[1]), torch.abs(om - CLIP_W[0]),
                  torch.abs(om - CLIP_W[1])]
        S, O = self.rollout(u, world, oc)
        for t in range(1, self.H + 1):
            x, y, v, th = S[t, 0], S[t, 1], S[t, 2], S[t, 3]
            e = v * torch.sin(th) - self.ts
            m.append(torch.abs(e * e - self.bound).reshape(1))
            if self.L > 1:
                f = torch.sort(((x - self.lane_x) * -1) ** 2 * 10).values
                m.append((f[1] - f[0]).reshape(1))
            ox, oy = O[t, :, 0], O[t, :, 1]
            nx, ny = (x - ox) / self.hx, (y - oy) / self.hy
            m += [torch.abs(1 - nx * nx), torch.abs(1 - ny * ny)]
            if self.C > 2:      # relative: the products carry relative rounding, and a lone nonzero one has gap 1
                pr = torch.sort(self._bump(x, ox - self.hx, ox + self.hx) * self._bump(y, oy - self.hy, oy + self.hy),
                                descending=True).values
                m.append(torch.where(pr[0] > 0, (pr[0] - pr[1]) / torch.where(pr[0] > 0, pr[0], 1.0), inf).reshape(1))
            for z in (x, -x):
                q = z - self.thr_lo
                m.append(torch.stack([torch.abs(q), torch.abs(self.thr_w - q)]))
            # abs's branch matters only where the fence's ramp factor is nonzero
            m.append(torch.where(self._threshold(x) + self._threshold(-x) > 0, torch.abs(x), inf).reshape(1))
        return torch.min(torch.cat(m))

    def sgd_margin(self, world, w, oc, s, n_iter: int):
        """branch_margin over the iterates the reverse pass differentiates at (u^0 .. u^{N-1}); inf for N = 0."""
        its = self.sgd_iterates(world, w, oc, s, n_iter)
        ms = [self.branch_margin(its[n], world, oc, computed=True) for n in range(n_iter)]
        return torch.min(torch.stack(ms)) if ms else self._c(float("inf"))

    # ---- batches: numpy in, numpy out ---------------------------------------------------------------------------------
    def _t(self, a, shape):
        return torch.as_tensor(np.array(a, np.float64).reshape(shape), dtype=self.dtype)

    def _args(self, B, u=None, world=None, w=None, oc=None):
        """numpy batches -> tensors; oc [B|1][C-1][H][2] or None (zeros: the model ignores it)."""
        out = {}
        if u is not None:
            out["u"] = self._t(u, (B, 2 * self.H))
        if world is not None:
            out["world"] = self._t(world, (B, self.C, 4))
        if w is not None:
            out["w"] = self._t(w, (B, self.K))
        oc = np.zeros((1, self.C - 1, self.H, 2)) if oc is None else np.asarray(oc, np.float64)
        out["oc"] = self._t(np.broadcast_to(oc.reshape(-1, self.C - 1, self.H, 2), (B, self.C - 1, self.H, 2)),
                            (B, self.C - 1, self.H, 2))
        return out

    def _map(self, fn, *args):
        """vmap fn over the leading axis of every argument, in chunks; -> numpy (a tuple for tuple results)."""
        B = args[0].shape[0]
        outs = []
        for i in range(0, B, self.chunk):
            r = vmap(fn)(*(a[i:i + self.chunk] for a in args))
            outs.append(r if isinstance(r, tuple) else (r,))
        res = tuple(torch.cat([o[j] for o in outs]).detach().numpy() for j in range(len(outs[0])))
        return res if len(res) > 1 else res[0]

    def batch_phi_sum(self, world, u, oc=None):
        a = self._args(len(world), u=u, world=world, oc=oc)
        return self._map(self.phi_sum, a["u"], a["world"], a["oc"])

    def batch_feature_jacobian(self, world, u, oc=None):
        a = self._args(len(world), u=u, world=world, oc=oc)
        return self._map(self.feature_jacobian, a["u"], a["world"], a["oc"])

    def batch_feature_hessian(self, world, u, oc=None):
        a = self._args(len(world), u=u, world=world, oc=oc)
        return self._map(self.feature_hessian, a["u"], a["world"], a["oc"])

    def batch_reward(self, world, u, w, oc=None):
        """-> (reward [B], grad_u [B][2H])."""
        a = self._args(len(world), u=u, world=world, w=w, oc=oc)
        return self._map(lambda *x: (self.reward(*x), self.grad_u(*x)), a["u"], a["world"], a["w"], a["oc"])

    def batch_hessian_u(self, world, u, w, oc=None):
        a = self._args(len(world), u=u, world=world, w=w, oc=oc)
        return self._map(self.hessian_u, a["u"], a["world"], a["w"], a["oc"])

    def batch_branch_margin(self, world, u, oc=None):
        a = self._args(len(world), u=u, world=world, oc=oc)
        return self._map(self.branch_margin, a["u"], a["world"], a["oc"])

    def batch_sgd_iterates(self, world, w, starts, n_iter: int, oc=None):
        a = self._args(len(world), world=world, w=w, oc=oc)
        s = torch.as_tensor(np.asarray(starts, np.int64))
        return self._map(lambda x, w_, o, s_: self.sgd_iterates(x, w_, o, s_, n_iter), a["world"], a["w"], a["oc"], s)

    def batch_sgd_vjp(self, world, w, starts, n_iter: int, plan_bar, oc=None):
        """-> (weights_bar [B][K], world_bar [B][C][4], margin [B]) for start starts[b] of problem b."""
        B = len(world)
        a = self._args(B, world=world, w=w, oc=oc)
        s = torch.as_tensor(np.asarray(starts, np.int64))
        pb = self._t(plan_bar, (B, 2 * self.H))

        def one(x, w_, o, s_, pb_):
            wb, xb = self.sgd_vjp(x, w_, o, s_, n_iter, pb_)
            return wb, xb, self.sgd_margin(x, w_, o, s_, n_iter)
        return self._map(one, a["world"], a["w"], a["oc"], s, pb)

    def batch_sgd_vjp_along(self, world, w, starts, its, plan_bar, oc=None):
        """-> (weights_bar [B][K], world_bar [B][C][4]) along the iterates its [B][N][2H]."""
        B = len(world)
        a = self._args(B, world=world, w=w, oc=oc)
        s = torch.as_tensor(np.asarray(starts, np.int64))
        it = torch.as_tensor(np.array(its, np.float64), dtype=self.dtype)
        pb = self._t(plan_bar, (B, 2 * self.H))
        return self._map(lambda x, w_, o, s_, i_, p_: self.sgd_vjp_along(x, w_, o, s_, i_, p_), a["world"], a["w"],
                         a["oc"], s, it, pb)

    def implicit_vjp(self, world, w, plan, plan_bar, oc=None):
        """The implicit-function VJP of ocd_b200.h at the given plans, batched: with A the controls inside the clip box,
        z_A = H_AA^{-1} plan_bar_A (solved in float64 whatever the dtype), theta_bar = -z_A . dG_A/dtheta.
        -> (weights_bar [B][K], world_bar [B][C][4], cond(H_AA) [B]; inf where H_AA is exactly singular)."""
        B = len(world)
        a = self._args(B, u=plan, world=world, w=w, oc=oc)
        Hs = self._map(self.hessian_u, a["u"], a["world"], a["w"], a["oc"])
        Gw, Gx = self._map(self.grad_u_mixed, a["u"], a["world"], a["w"], a["oc"])
        u = np.asarray(plan, np.float64).reshape(B, -1)
        pb = np.asarray(plan_bar, np.float64).reshape(B, -1)
        wb, xb, cond = np.zeros((B, self.K)), np.zeros((B, self.C, 4)), np.zeros(B)
        for b in range(B):
            act = np.ones(u.shape[1], bool)
            act[0::2] = (u[b, 0::2] >= CLIP_A[0]) & (u[b, 0::2] <= CLIP_A[1])
            act[1::2] = (u[b, 1::2] >= CLIP_W[0]) & (u[b, 1::2] <= CLIP_W[1])
            if not act.any():
                continue
            Haa = Hs[b][np.ix_(act, act)].astype(np.float64)
            cond[b] = np.linalg.cond(Haa)
            if not np.isfinite(cond[b]):
                cond[b] = np.inf
                continue
            z = np.linalg.solve(Haa, pb[b, act])
            wb[b] = -z @ Gw[b][act].astype(np.float64)
            xb[b] = -np.tensordot(z, Gx[b][act].astype(np.float64), axes=1)
        return wb, xb, cond
