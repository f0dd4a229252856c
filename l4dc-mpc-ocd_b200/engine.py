"""Batched MPC engine: Python front-end of the C ABI (``include/ocd_b200.h``).

torch is used for device memory and streams only; every number is produced by the CUDA kernels
in ``csrc/``.  Arrays cross the ABI in structure-of-arrays layout with the batch index fastest
(``[C][4][B]``); the ``*_soa`` methods take and return that layout untouched, the plain methods
accept the natural ``[B, C, 4]`` shapes and transpose on the device.

What each call replaces in the reference (paths relative to the reference checkout):
  solve      NaivePlanner.generate_plan             interact_drive/planner/naive_planner.py:81-164
  reward     NaivePlanner.reward_func (+ d/dcontrols) interact_drive/planner/naive_planner.py:32-79
  features   ThreeLaneTestCar.features              experiments/merging.py:32-83
  dynamics   car_dynamics_step / Car.step           interact_drive/simulation_utils.py:9-21
  episodes   MPC_ORD.eval_weights_for_init's loop   interact_drive/reward_design/mpc_ord.py:87-103
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Optional, Sequence

import numpy as np
import torch

from . import _native as N

MATH_FAST, MATH_PRECISE = 0, 1
OPT_SGD, OPT_LBFGS = 0, 1


@dataclass
class PlannerParams:
    """Planner + world constants (``ocd_params``)."""
    H: int = 5
    C: int = 2
    lane_x: Sequence[float] = (-0.1, 0.0, 0.1)
    n_iter: int = 100
    num_lanes: int = 3
    other_mode: int = 0            # 0: other cars keep velocity; 1: known controls
    extra_inits: bool = False
    math_mode: int = MATH_FAST
    optimizer: int = OPT_SGD       # OPT_LBFGS: opt-in L-BFGS (H <= 16), n_iter = maximum iterations
    lr: float = 0.1
    dt: float = 0.1
    friction: float = 0.2
    target_speed: float = 1.0

    @property
    def L(self) -> int:
        return len(self.lane_x)

    @property
    def K(self) -> int:
        return self.L + 4

    @property
    def S(self) -> int:
        return 6 if self.extra_inits else 3

    def c_struct(self) -> N.ocd_params:
        if self.L > N.MAX_LANES:
            raise ValueError(f"at most {N.MAX_LANES} lanes are supported, got {self.L}")
        p = N.ocd_params()
        p.H, p.C, p.L, p.n_iter = int(self.H), int(self.C), self.L, int(self.n_iter)
        p.num_lanes, p.other_mode = int(self.num_lanes), int(self.other_mode)
        p.extra_inits, p.math_mode = int(bool(self.extra_inits)), int(self.math_mode)
        p.optimizer, p.reserved = int(self.optimizer), 0
        p.lr, p.dt, p.friction, p.target_speed = float(self.lr), float(self.dt), float(self.friction), \
            float(self.target_speed)
        for i, x in enumerate(self.lane_x):
            p.lane_x[i] = float(x)
        return p


@dataclass
class Scenario:
    """Scripted cars (cars 1..C-1) and the replanning teleport (``ocd_scenario``)."""
    init_state: Sequence[Sequence[float]] = ()
    kind: Sequence[int] = ()                 # 0 fixed control / fixed velocity, 1 fixed plan
    friction: Sequence[float] = ()
    control: Sequence[Sequence[float]] = ()  # fixed control / default control
    plan: Sequence[Sequence[Sequence[float]]] = ()
    critical_t: int = 0
    teleport_state: Sequence[float] = (10.0, 0.0, 0.0, 0.0)

    def c_struct(self) -> N.ocd_scenario:
        n = len(self.init_state)
        if n > N.MAX_OTHER:
            raise ValueError(f"at most {N.MAX_OTHER} other cars are supported, got {n}")
        s = N.ocd_scenario()
        s.n_other, s.critical_t = n, int(self.critical_t)
        for j in range(n):
            s.kind[j] = int(self.kind[j])
            s.friction[j] = float(self.friction[j])
            for c in range(4):
                s.init_state[j][c] = float(self.init_state[j][c])
            for c in range(2):
                s.control[j][c] = float(self.control[j][c])
            pl = self.plan[j] if j < len(self.plan) else ()
            if len(pl) > N.MAX_PLAN:
                raise ValueError(f"plans longer than {N.MAX_PLAN} steps are not supported")
            s.plan_len[j] = len(pl)
            for t, u in enumerate(pl):
                s.plan[j][t][0], s.plan[j][t][1] = float(u[0]), float(u[1])
        for c in range(4):
            s.teleport_state[c] = float(self.teleport_state[c])
        return s


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _check_soa(name: str, t: Optional[torch.Tensor], dtype, device, shape) -> None:
    """The *_soa entry points hand raw device pointers to the kernels: a tensor of another dtype, device, layout or
    shape would be reinterpreted, so it is refused here (ValueError, like the reference's shape checks)."""
    if t is None:
        return
    if not torch.is_tensor(t) or t.dtype != dtype or t.device != device or not t.is_contiguous() \
            or tuple(t.shape) != tuple(shape):
        got = (tuple(t.shape), t.dtype, t.device, t.is_contiguous()) if torch.is_tensor(t) else type(t)
        raise ValueError(f"{name} must be a contiguous {dtype} tensor of shape {tuple(shape)} on {device}, got {got}")


FORM_NAMES = {N.FORM_THROUGHPUT: "throughput", N.FORM_LATENCY: "latency", N.FORM_WIDE: "wide",
              N.FORM_TIME_PARALLEL: "time-parallel"}


def kernel_form(p: "PlannerParams", B: int, episode: bool = False) -> str:
    """Which form of the planner kernel a batch of B problems (or B episode worlds) would run -- host logic, needs
    no GPU (`ocd_kernel_form`)."""
    ps = p.c_struct()
    rc = N.lib.ocd_kernel_form(C.addressof(ps), int(B), int(bool(episode)))
    if rc < 0:
        N.check(rc, "ocd_kernel_form")
    return FORM_NAMES[rc]


def device_count() -> int:
    return int(N.lib.ocd_device_count())


class Engine:
    """One engine per device.  All methods enqueue on torch's current stream for that device and
    return device tensors without synchronising."""

    def __init__(self, device: int | str | torch.device = 0):
        if device_count() < 1:
            raise N.OcdCudaError("no CUDA device visible: the batched MPC engine has no CPU fallback")
        self.device = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
        if self.device.type != "cuda":
            raise N.OcdCudaError(f"the batched MPC engine runs on CUDA devices only, not {self.device}")
        self._kernel_launches = 0

    # -- helpers -------------------------------------------------------------------------------
    @property
    def kernel_launches(self) -> int:
        """Number of engine kernels launched through this object (bench.py's gpu_launches)."""
        return self._kernel_launches

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _f32(self, x, shape=None) -> torch.Tensor:
        t = torch.as_tensor(x, dtype=torch.float32, device=self.device)
        if shape is not None:
            t = t.reshape(shape)
        return t.contiguous()

    def _i32(self, x, shape=None) -> torch.Tensor:
        t = torch.as_tensor(x, dtype=torch.int32, device=self.device)
        if shape is not None:
            t = t.reshape(shape)
        return t.contiguous()

    def _weights(self, p: PlannerParams, weights, weight_idx, B):
        """-> (weights [K][Bw] on device, Bw, weight_idx [B] or None)."""
        w = torch.as_tensor(weights, dtype=torch.float32, device=self.device)
        if w.dim() == 1:
            w = w.reshape(1, -1)
        if w.shape[-1] != p.K:
            raise ValueError(f"weights must have {p.K} entries per vector, got shape {tuple(w.shape)}")
        Bw = w.shape[0]
        idx = None
        if weight_idx is not None:
            if not torch.is_tensor(weight_idx) or not weight_idx.is_cuda:
                # host-side indices are checked before the upload (device-resident ones are clamped by the kernels:
                # checking them here would cost a synchronising copy)
                wi = np.asarray(weight_idx.cpu() if torch.is_tensor(weight_idx) else weight_idx)
                if wi.size and (wi.min() < 0 or wi.max() >= Bw):
                    raise ValueError(f"weight_idx must lie in [0, {Bw}), got [{wi.min()}, {wi.max()}]")
            idx = self._i32(weight_idx, (B,))
        elif Bw not in (1, B):
            raise ValueError(f"{Bw} weight vectors for {B} problems need a weight_idx")
        return w.t().contiguous(), Bw, idx

    # -- structure-of-arrays entry points (no reshuffling, what bench.py times) ---------------------
    def solve_soa(self, p: PlannerParams, world, weights, Bw: int, weight_idx=None, other_controls=None,
                  Bo: int = 0, cur_speed=None, all_plans: bool = False, out=None):
        """world [C][4][B], weights [K][Bw], other_controls [C-1][H][2][Bo] -> plan [H][2][B],
        losses [S][B], best [B] (+ all_plans [S][H][2][B])."""
        B = world.shape[-1]
        dev = self.device
        f32, i32 = torch.float32, torch.int32
        _check_soa("world", world, f32, dev, (p.C, 4, B))
        _check_soa("weights", weights, f32, dev, (p.K, Bw))
        _check_soa("weight_idx", weight_idx, i32, dev, (B,))
        _check_soa("cur_speed", cur_speed, f32, dev, (B,))
        if p.other_mode == 1:
            if other_controls is None or Bo not in (1, B):
                raise ValueError("other_mode=1 needs other_controls [C-1][H][2][Bo] with Bo in (1, B)")
            _check_soa("other_controls", other_controls, f32, dev, (p.C - 1, p.H, 2, Bo))
        if out is not None:
            _check_soa("out['plan']", out["plan"], f32, dev, (p.H, 2, B))
            _check_soa("out['losses']", out["losses"], f32, dev, (p.S, B))
            _check_soa("out['best']", out["best"], i32, dev, (B,))
            _check_soa("out['all_plans']", out.get("all_plans"), f32, dev, (p.S, p.H, 2, B))
        if out is None:
            out = dict(plan=torch.empty((p.H, 2, B), dtype=torch.float32, device=dev),
                       losses=torch.empty((p.S, B), dtype=torch.float32, device=dev),
                       best=torch.empty((B,), dtype=torch.int32, device=dev))
            if all_plans:
                out["all_plans"] = torch.empty((p.S, p.H, 2, B), dtype=torch.float32, device=dev)
        ps = p.c_struct()
        with torch.cuda.device(dev):
            rc = N.lib.ocd_solve_batch(C.addressof(ps), _ptr(world), _ptr(other_controls), Bo, _ptr(weights), Bw,
                                       _ptr(weight_idx), _ptr(cur_speed), _ptr(out["plan"]), _ptr(out["losses"]),
                                       _ptr(out["best"]), _ptr(out.get("all_plans")), B, self._stream())
        N.check(rc, "ocd_solve_batch")
        self._kernel_launches += 1 if B else 0
        return out

    def solve_vjp_soa(self, p: PlannerParams, world, weights, Bw: int, best, plan_bar, weight_idx=None,
                      other_controls=None, Bo: int = 0, cur_speed=None, world_bar: bool = True):
        """Vector-Jacobian product of solve_soa's plan (``ocd_solve_vjp_batch``): the same inputs, solve_soa's `best`
        and plan_bar [H][2][B] = d loss / d plan -> dict(weights_bar [K][B]: d loss / d (problem b's weight vector),
        world_bar [C][4][B] (with world_bar=True)).  Rows are per problem; problems sharing a weight vector are not
        summed here.  The workspace (n_iter * H * 2 * B floats) is allocated on the device for the call."""
        B = world.shape[-1]
        dev = self.device
        f32, i32 = torch.float32, torch.int32
        _check_soa("world", world, f32, dev, (p.C, 4, B))
        _check_soa("weights", weights, f32, dev, (p.K, Bw))
        _check_soa("weight_idx", weight_idx, i32, dev, (B,))
        _check_soa("cur_speed", cur_speed, f32, dev, (B,))
        _check_soa("best", best, i32, dev, (B,))
        _check_soa("plan_bar", plan_bar, f32, dev, (p.H, 2, B))
        if p.other_mode == 1:
            if other_controls is None or Bo not in (1, B):
                raise ValueError("other_mode=1 needs other_controls [C-1][H][2][Bo] with Bo in (1, B)")
            _check_soa("other_controls", other_controls, f32, dev, (p.C - 1, p.H, 2, Bo))
        ps = p.c_struct()
        nbytes = C.c_size_t(0)
        N.check(N.lib.ocd_solve_vjp_workspace_bytes(C.addressof(ps), B, C.byref(nbytes)), "ocd_solve_vjp_workspace_bytes")
        ws = torch.empty((nbytes.value // 4,), dtype=f32, device=dev)
        out = dict(weights_bar=torch.empty((p.K, B), dtype=f32, device=dev))
        if world_bar:
            out["world_bar"] = torch.empty((p.C, 4, B), dtype=f32, device=dev)
        with torch.cuda.device(dev):
            rc = N.lib.ocd_solve_vjp_batch(C.addressof(ps), _ptr(world), _ptr(other_controls), Bo, _ptr(weights), Bw,
                                           _ptr(weight_idx), _ptr(cur_speed), _ptr(best), _ptr(plan_bar),
                                           _ptr(out["weights_bar"]), _ptr(out.get("world_bar")), _ptr(ws),
                                           nbytes.value, B, self._stream())
        N.check(rc, "ocd_solve_vjp_batch")
        self._kernel_launches += 1 if B else 0
        return out

    def episodes_soa(self, p: PlannerParams, sc: Scenario, robot_init, plan_weights, Bw: int, true_weights, T: int,
                     weight_idx=None, other_init=None, unlucky_idx=None, t0: int = 0, trace: bool = False,
                     final_world: bool = False, out=None):
        """robot_init [4][B], plan_weights [K][Bw], true_weights [K] -> returns [B]
        (+ controls [T][2][B], best [T][B], states [T][C][4][B], final_world [C][4][B])."""
        B = robot_init.shape[-1]
        dev = self.device
        f32, i32 = torch.float32, torch.int32
        _check_soa("robot_init", robot_init, f32, dev, (4, B))
        _check_soa("plan_weights", plan_weights, f32, dev, (p.K, Bw))
        _check_soa("true_weights", true_weights, f32, dev, (p.K,))
        _check_soa("weight_idx", weight_idx, i32, dev, (B,))
        _check_soa("other_init", other_init, f32, dev, (p.C - 1, 4, B))
        _check_soa("unlucky_idx", unlucky_idx, i32, dev, (B,))
        if out is not None:
            _check_soa("out['returns']", out["returns"], f32, dev, (B,))
            _check_soa("out['controls']", out.get("controls"), f32, dev, (T, 2, B))
            _check_soa("out['best']", out.get("best"), i32, dev, (T, B))
            _check_soa("out['states']", out.get("states"), f32, dev, (T, p.C, 4, B))
            _check_soa("out['final_world']", out.get("final_world"), f32, dev, (p.C, 4, B))
        if out is None:
            out = dict(returns=torch.empty((B,), dtype=torch.float32, device=dev))
            if trace:
                out["controls"] = torch.empty((T, 2, B), dtype=torch.float32, device=dev)
                out["best"] = torch.empty((T, B), dtype=torch.int32, device=dev)
                out["states"] = torch.empty((T, p.C, 4, B), dtype=torch.float32, device=dev)
            if final_world:
                out["final_world"] = torch.empty((p.C, 4, B), dtype=torch.float32, device=dev)
        ps, ss = p.c_struct(), sc.c_struct()
        with torch.cuda.device(dev):
            rc = N.lib.ocd_episode_batch(C.addressof(ps), C.addressof(ss), _ptr(robot_init), _ptr(other_init),
                                         _ptr(plan_weights), Bw, _ptr(weight_idx), _ptr(true_weights),
                                         _ptr(unlucky_idx), int(t0), int(T), _ptr(out["returns"]),
                                         _ptr(out.get("controls")), _ptr(out.get("best")), _ptr(out.get("states")),
                                         _ptr(out.get("final_world")), B, self._stream())
        N.check(rc, "ocd_episode_batch")
        self._kernel_launches += 1 if B else 0
        return out

    # -- natural-shape entry points ------------------------------------------------------------
    def _world(self, p: PlannerParams, world) -> torch.Tensor:
        w = torch.as_tensor(world, dtype=torch.float32, device=self.device)
        if w.dim() == 2:
            w = w.unsqueeze(0)
        if w.dim() != 3 or w.shape[1] != p.C or w.shape[2] != 4:
            raise ValueError(f"world state must have shape [B, {p.C}, 4], got {tuple(w.shape)}")
        return w.permute(1, 2, 0).contiguous()

    def _other_controls(self, p: PlannerParams, other_controls, B):
        if p.other_mode != 1:
            return None, 0
        if other_controls is None:
            raise ValueError("other_mode=1 needs other_controls")
        oc = torch.as_tensor(other_controls, dtype=torch.float32, device=self.device)
        if oc.dim() == 3:
            oc = oc.unsqueeze(0)
        if oc.dim() != 4 or tuple(oc.shape[1:]) != (p.C - 1, p.H, 2) or oc.shape[0] not in (1, B):
            raise ValueError(f"other_controls must have shape [B|1, {p.C - 1}, {p.H}, 2], got {tuple(oc.shape)}")
        return oc.permute(1, 2, 3, 0).contiguous(), oc.shape[0]

    def solve(self, p: PlannerParams, world, weights, weight_idx=None, other_controls=None, cur_speed=None,
              all_plans: bool = False):
        """world [B, C, 4]; weights [K] | [Bw, K]; other_controls [B|1, C-1, H, 2] ->
        dict(plan [B, H, 2], losses [B, S], best [B] (+ all_plans [B, S, H, 2]))."""
        ws = self._world(p, world)
        B = ws.shape[-1]
        w, Bw, idx = self._weights(p, weights, weight_idx, B)
        oc, Bo = self._other_controls(p, other_controls, B)
        cs = None if cur_speed is None else self._f32(cur_speed, (B,))
        o = self.solve_soa(p, ws, w, Bw, idx, oc, Bo, cs, all_plans)
        res = dict(plan=o["plan"].permute(2, 0, 1).contiguous(), losses=o["losses"].t().contiguous(), best=o["best"])
        if all_plans:
            res["all_plans"] = o["all_plans"].permute(3, 0, 1, 2).contiguous()
        return res

    def reward(self, p: PlannerParams, world, controls, weights, weight_idx=None, other_controls=None,
               grad: bool = True):
        """world [B, C, 4]; controls [B, H, 2] -> reward [B] (and d reward / d controls [B, H, 2])."""
        ws = self._world(p, world)
        B = ws.shape[-1]
        u = torch.as_tensor(controls, dtype=torch.float32, device=self.device)
        if u.dim() == 2:
            u = u.unsqueeze(0)
        if tuple(u.shape) != (B, p.H, 2):
            raise ValueError(f"controls must have shape [{B}, {p.H}, 2], got {tuple(u.shape)}")
        us = u.permute(1, 2, 0).contiguous()
        w, Bw, idx = self._weights(p, weights, weight_idx, B)
        oc, Bo = self._other_controls(p, other_controls, B)
        R = torch.empty((B,), dtype=torch.float32, device=self.device)
        G = torch.empty((p.H, 2, B), dtype=torch.float32, device=self.device) if grad else None
        ps = p.c_struct()
        with torch.cuda.device(self.device):
            rc = N.lib.ocd_reward_grad_batch(C.addressof(ps), _ptr(ws), _ptr(us), _ptr(oc), Bo, _ptr(w), Bw, _ptr(idx),
                                             _ptr(R), _ptr(G), B, self._stream())
        N.check(rc, "ocd_reward_grad_batch")
        self._kernel_launches += 1 if B else 0
        return (R, G.permute(2, 0, 1).contiguous()) if grad else R

    def feature_jacobian(self, p: PlannerParams, world, controls, other_controls=None):
        """world [B, C, 4]; controls [B, H, 2] -> (phi_sum [B, K], jac [B, K, H, 2]): the horizon-summed
        features and their Jacobian with respect to the controls (row i = d sum_t phi_i / d u)."""
        ws = self._world(p, world)
        B = ws.shape[-1]
        u = torch.as_tensor(controls, dtype=torch.float32, device=self.device)
        if u.dim() == 2:
            u = u.unsqueeze(0)
        if tuple(u.shape) != (B, p.H, 2):
            raise ValueError(f"controls must have shape [{B}, {p.H}, 2], got {tuple(u.shape)}")
        us = u.permute(1, 2, 0).contiguous()
        oc, Bo = self._other_controls(p, other_controls, B)
        phi = torch.empty((p.K, B), dtype=torch.float32, device=self.device)
        jac = torch.empty((p.K, p.H, 2, B), dtype=torch.float32, device=self.device)
        ps = p.c_struct()
        with torch.cuda.device(self.device):
            rc = N.lib.ocd_feature_jacobian_batch(C.addressof(ps), _ptr(ws), _ptr(us), _ptr(oc), Bo, _ptr(phi),
                                                  _ptr(jac), B, self._stream())
        N.check(rc, "ocd_feature_jacobian_batch")
        self._kernel_launches += 1 if B else 0
        return phi.t().contiguous(), jac.permute(3, 0, 1, 2).contiguous()

    def feature_hessian(self, p: PlannerParams, world, controls, other_controls=None) -> torch.Tensor:
        """world [B, C, 4]; controls [B, H, 2] -> hess [B, K, 2H, 2H]: the Hessian of every horizon-summed feature
        with respect to the flattened controls (index 2 t + c).  The reward's Hessian is sum_k w_k hess[:, k]."""
        ws = self._world(p, world)
        B = ws.shape[-1]
        u = torch.as_tensor(controls, dtype=torch.float32, device=self.device)
        if u.dim() == 2:
            u = u.unsqueeze(0)
        if tuple(u.shape) != (B, p.H, 2):
            raise ValueError(f"controls must have shape [{B}, {p.H}, 2], got {tuple(u.shape)}")
        us = u.permute(1, 2, 0).contiguous()
        oc, Bo = self._other_controls(p, other_controls, B)
        n = 2 * p.H
        hess = torch.empty((p.K, n, n, B), dtype=torch.float32, device=self.device)
        ps = p.c_struct()
        with torch.cuda.device(self.device):
            rc = N.lib.ocd_feature_hessian_batch(C.addressof(ps), _ptr(ws), _ptr(us), _ptr(oc), Bo, _ptr(hess), B,
                                                 self._stream())
        N.check(rc, "ocd_feature_hessian_batch")
        self._kernel_launches += 1 if B else 0
        return hess.permute(3, 0, 1, 2).contiguous()

    def features(self, p: PlannerParams, world) -> torch.Tensor:
        """world [B, C, 4] -> phi [B, K]."""
        ws = self._world(p, world)
        B = ws.shape[-1]
        phi = torch.empty((p.K, B), dtype=torch.float32, device=self.device)
        ps = p.c_struct()
        with torch.cuda.device(self.device):
            rc = N.lib.ocd_features_batch(C.addressof(ps), _ptr(ws), _ptr(phi), B, self._stream())
        N.check(rc, "ocd_features_batch")
        self._kernel_launches += 1 if B else 0
        return phi.t().contiguous()

    def smooth(self, kind: int, z, p0: float, p1: float = 0.0) -> torch.Tensor:
        """_f / smooth_threshold / smooth_bump of interact_drive/math_utils.py at the points z."""
        zt = torch.as_tensor(z, dtype=torch.float32, device=self.device)
        shape = zt.shape
        zt = zt.reshape(-1).contiguous()
        out = torch.empty_like(zt)
        with torch.cuda.device(self.device):
            rc = N.lib.ocd_smooth_batch(int(kind), _ptr(zt), float(p0), float(p1), _ptr(out), zt.numel(), self._stream())
        N.check(rc, "ocd_smooth_batch")
        self._kernel_launches += 1 if zt.numel() else 0
        return out.reshape(shape)

    def dynamics(self, state, control, dt: float, friction) -> torch.Tensor:
        """state [B, 4], control [B, 2], friction scalar or [B] -> next state [B, 4]."""
        s = torch.as_tensor(state, dtype=torch.float32, device=self.device)
        u = torch.as_tensor(control, dtype=torch.float32, device=self.device)
        if s.dim() == 1:
            s, u = s.unsqueeze(0), u.reshape(1, -1)
        if s.dim() != 2 or s.shape[1] != 4 or u.dim() != 2 or tuple(u.shape) != (s.shape[0], 2):
            # same failure the reference raises for malformed shapes (simulation_utils.py:110-115)
            raise ValueError(f"expected state [B, 4] and control [B, 2], got {tuple(s.shape)} and {tuple(u.shape)}")
        B = s.shape[0]
        ss, us = s.t().contiguous(), u.t().contiguous()
        fb, f0 = None, 0.0
        if np.ndim(friction) == 0 and not torch.is_tensor(friction):
            f0 = float(friction)
        else:
            fb = self._f32(friction, (B,))
        out = torch.empty_like(ss)
        with torch.cuda.device(self.device):
            rc = N.lib.ocd_dynamics_step_batch(_ptr(ss), _ptr(us), float(dt), f0, _ptr(fb), _ptr(out), B,
                                               self._stream())
        N.check(rc, "ocd_dynamics_step_batch")
        self._kernel_launches += 1 if B else 0
        return out.t().contiguous()

    def episodes(self, p: PlannerParams, sc: Scenario, robot_init, plan_weights, true_weights, T: int,
                 weight_idx=None, other_init=None, unlucky_idx=None, t0: int = 0, trace: bool = False,
                 final_world: bool = False):
        """robot_init [B, 4]; plan_weights [K] | [Bw, K]; true_weights [K] -> dict(returns [B], and with
        trace: controls [B, T, 2], best [B, T], states [B, T, C, 4]; final_world [B, C, 4])."""
        ri = torch.as_tensor(robot_init, dtype=torch.float32, device=self.device)
        if ri.dim() == 1:
            ri = ri.unsqueeze(0)
        if ri.dim() != 2 or ri.shape[1] != 4:
            raise ValueError(f"robot_init must have shape [B, 4], got {tuple(ri.shape)}")
        B = ri.shape[0]
        ris = ri.t().contiguous()
        w, Bw, idx = self._weights(p, plan_weights, weight_idx, B)
        tw = self._f32(true_weights, (p.K,))
        oi = None
        if other_init is not None:
            o = torch.as_tensor(other_init, dtype=torch.float32, device=self.device)
            if tuple(o.shape) != (B, p.C - 1, 4):
                raise ValueError(f"other_init must have shape [{B}, {p.C - 1}, 4], got {tuple(o.shape)}")
            oi = o.permute(1, 2, 0).contiguous()
        ul = None if unlucky_idx is None else self._i32(unlucky_idx, (B,))
        o = self.episodes_soa(p, sc, ris, w, Bw, tw, T, idx, oi, ul, t0, trace, final_world)
        res = dict(returns=o["returns"])
        if trace:
            res["controls"] = o["controls"].permute(2, 0, 1).contiguous()
            res["best"] = o["best"].t().contiguous()
            res["states"] = o["states"].permute(3, 0, 1, 2).contiguous()
        if final_world:
            res["final_world"] = o["final_world"].permute(2, 0, 1).contiguous()
        return res

    def fp32_peak(self, iters: int = 4096) -> float:
        """Measured FP32 FMA throughput (FLOP/s) of this device: bench.py's roofline denominator."""
        fl = C.c_double(0.0)
        with torch.cuda.device(self.device):
            rc = N.lib.ocd_fp32_peak(int(iters), C.byref(fl), self._stream())
        N.check(rc, "ocd_fp32_peak")
        return float(fl.value)


class HostContext:
    """``ocd_ctx``: the host-buffer path of the C ABI (numpy in, numpy out, copies inside)."""

    def __init__(self, device: int = 0):
        h = C.c_void_p()
        N.check(N.lib.ocd_ctx_create(int(device), C.byref(h)), "ocd_ctx_create")
        self._h = h

    def close(self):
        if self._h:
            N.lib.ocd_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def pinned_empty(shape, dtype=np.float32) -> np.ndarray:
        """A page-locked host array: the copy engines read / write it in place, so the host-buffer
        calls skip their staging copies (pageable arrays work too, through a pinned staging area)."""
        t = torch.empty(tuple(shape), dtype=torch.float32 if np.dtype(dtype) == np.float32 else torch.int32,
                        pin_memory=True)
        return t.numpy()          # the array keeps the pinned storage alive (ndarray.base), and frees it with itself

    @staticmethod
    def register(array: np.ndarray) -> np.ndarray:
        """Page-lock an ordinary numpy array in place (ocd_host_register): a caller that reuses its input / output
        arrays registers them once and the host-buffer calls then copy from / into them directly, like arrays from
        pinned_empty -- no staging memcpy.  Call unregister(array) before the array is freed."""
        if not (isinstance(array, np.ndarray) and array.flags["C_CONTIGUOUS"]):
            raise ValueError("register needs a C-contiguous numpy array")
        N.check(N.lib.ocd_host_register(array.ctypes.data, array.nbytes), "ocd_host_register")
        return array

    @staticmethod
    def unregister(array: np.ndarray) -> None:
        N.check(N.lib.ocd_host_unregister(array.ctypes.data), "ocd_host_unregister")

    def solve_soa(self, p: PlannerParams, world: np.ndarray, weights: np.ndarray, weight_idx=None,
                  other_controls=None, cur_speed=None, out=None):
        """Host SoA arrays: world [C][4][B], weights [K][Bw] -> plan [H][2][B], losses [S][B], best [B].
        `out` may hold preallocated (ideally pinned) plan / losses / best arrays."""
        world = np.ascontiguousarray(world, np.float32)
        weights = np.ascontiguousarray(weights, np.float32)
        B, Bw = world.shape[-1], weights.shape[-1]
        idx = None if weight_idx is None else np.ascontiguousarray(weight_idx, np.int32)
        oc = None if other_controls is None else np.ascontiguousarray(other_controls, np.float32)
        Bo = 0 if oc is None else oc.shape[-1]
        cs = None if cur_speed is None else np.ascontiguousarray(cur_speed, np.float32)
        if out is None:
            out = dict(plan=np.empty((p.H, 2, B), np.float32), losses=np.empty((p.S, B), np.float32),
                       best=np.empty((B,), np.int32))
        plan, losses, best = out["plan"], out["losses"], out["best"]
        if plan.shape != (p.H, 2, B) or losses.shape != (p.S, B) or best.shape != (B,) or \
                plan.dtype != np.float32 or losses.dtype != np.float32 or best.dtype != np.int32 or \
                not (plan.flags.c_contiguous and losses.flags.c_contiguous and best.flags.c_contiguous):
            raise ValueError("out arrays must be C-contiguous plan [H,2,B] f32, losses [S,B] f32, best [B] i32")
        ps = p.c_struct()
        vp = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
        rc = N.lib.ocd_solve_batch_host(self._h, C.addressof(ps), vp(world), vp(oc), Bo, vp(weights), Bw, vp(idx),
                                        vp(cs), vp(plan), vp(losses), vp(best), B)
        N.check(rc, "ocd_solve_batch_host")
        return dict(plan=plan, losses=losses, best=best)

    def solve_first_soa(self, p: PlannerParams, world: np.ndarray, weights: np.ndarray, weight_idx=None,
                        other_controls=None, cur_speed=None, out=None, losses: bool = True, best: bool = True):
        """The receding-horizon caller's solve (`ocd_solve_first_host`): only plan[0] comes back.
        Host SoA arrays in; -> dict(first [2][B] (+ losses [S][B], best [B])).  `out` may hold preallocated arrays."""
        world = np.ascontiguousarray(world, np.float32)
        weights = np.ascontiguousarray(weights, np.float32)
        B, Bw = world.shape[-1], weights.shape[-1]
        idx = None if weight_idx is None else np.ascontiguousarray(weight_idx, np.int32)
        oc = None if other_controls is None else np.ascontiguousarray(other_controls, np.float32)
        Bo = 0 if oc is None else oc.shape[-1]
        cs = None if cur_speed is None else np.ascontiguousarray(cur_speed, np.float32)
        if out is None:
            out = dict(first=np.empty((2, B), np.float32))
            if losses:
                out["losses"] = np.empty((p.S, B), np.float32)
            if best:
                out["best"] = np.empty((B,), np.int32)
        first, lo, be = out["first"], out.get("losses"), out.get("best")
        ok = first.shape == (2, B) and first.dtype == np.float32 and first.flags.c_contiguous
        ok = ok and (lo is None or (lo.shape == (p.S, B) and lo.dtype == np.float32 and lo.flags.c_contiguous))
        ok = ok and (be is None or (be.shape == (B,) and be.dtype == np.int32 and be.flags.c_contiguous))
        if not ok:
            raise ValueError("out arrays must be C-contiguous first [2,B] f32, losses [S,B] f32, best [B] i32")
        ps = p.c_struct()
        vp = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
        rc = N.lib.ocd_solve_first_host(self._h, C.addressof(ps), vp(world), vp(oc), Bo, vp(weights), Bw, vp(idx),
                                        vp(cs), vp(first), vp(lo), vp(be), B)
        N.check(rc, "ocd_solve_first_host")
        return out

    def episodes_soa(self, p: PlannerParams, sc: Scenario, robot_init: np.ndarray, plan_weights: np.ndarray,
                     true_weights: np.ndarray, T: int, weight_idx=None, other_init=None, unlucky_idx=None,
                     t0: int = 0, final_world: bool = False, structs=None):
        """Host SoA arrays: robot_init [4][B], plan_weights [K][Bw], true_weights [K] -> returns [B]
        (with final_world=True: (returns, final world [C][4][B])).  `structs`: a cached (ocd_params, ocd_scenario) pair
        for callers that make the same call over and over (MPC_ORD)."""
        ri = np.ascontiguousarray(robot_init, np.float32)
        w = np.ascontiguousarray(plan_weights, np.float32)
        tw = np.ascontiguousarray(true_weights, np.float32)
        B, Bw = ri.shape[-1], w.shape[-1]
        idx = None if weight_idx is None else np.ascontiguousarray(weight_idx, np.int32)
        oi = None if other_init is None else np.ascontiguousarray(other_init, np.float32)
        ul = None if unlucky_idx is None else np.ascontiguousarray(unlucky_idx, np.int32)
        ret = np.empty((B,), np.float32)
        fw = np.empty((p.C, 4, B), np.float32) if final_world else None
        ps, ss = structs if structs is not None else (p.c_struct(), sc.c_struct())
        vp = lambda a: None if a is None else a.ctypes.data          # plain address: argtypes make it a void pointer
        rc = N.lib.ocd_episode_batch_host(self._h, C.addressof(ps), C.addressof(ss), vp(ri), vp(oi), vp(w), Bw,
                                          vp(idx), vp(tw), vp(ul), int(t0), int(T), vp(ret), vp(fw), B)
        N.check(rc, "ocd_episode_batch_host")
        return (ret, fw) if final_world else ret
