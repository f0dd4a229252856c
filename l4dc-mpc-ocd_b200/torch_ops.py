"""The two planner entry points as PyTorch custom ops (``torch.ops.ocd_b200.solve`` /
``torch.ops.ocd_b200.episodes``) and their reverse passes (``torch.ops.ocd_b200.solve_vjp`` for SGD plans and
``torch.ops.ocd_b200.solve_implicit_vjp`` for L-BFGS plans, which make up
``solve``'s autograd formula: gradients of the plan reach ``world`` and ``weights``; ``torch.ops.ocd_b200.episodes_vjp``
(SGD) or ``torch.ops.ocd_b200.episodes_implicit_vjp`` (L-BFGS) with ``episodes_trace``, ``episodes``' autograd formula:
gradients of the returns reach ``robot_init``,
``plan_weights`` and ``true_weights``): device tensors in,
device tensors out, launched on the current stream through the same C ABI as everything else.  Registering them makes the engine usable from code that
composes torch ops (and gives them fake-tensor shape functions); there is deliberately no CPU kernel --
calling them with CPU tensors is an error, not a fallback.

Tensors are in the ABI's structure-of-arrays layout (batch index last).  The planner constants travel
as a flat list of numbers (see ``pack_params``) because custom-op schemas only carry tensors and scalars.
"""
from __future__ import annotations

from typing import List, Optional, Tuple

import torch

from .engine import Engine, PlannerParams, Scenario

_engines = {}


def _engine(t: torch.Tensor) -> Engine:
    if not t.is_cuda:
        raise RuntimeError("ocd_b200 ops run on CUDA tensors only (the engine has no CPU fallback)")
    idx = t.device.index if t.device.index is not None else torch.cuda.current_device()
    if idx not in _engines:
        _engines[idx] = Engine(idx)
    return _engines[idx]


def pack_params(p: PlannerParams) -> List[float]:
    """PlannerParams -> flat list understood by the ops."""
    return [float(p.H), float(p.C), float(p.n_iter), float(p.num_lanes), float(p.other_mode), float(bool(p.extra_inits)),
            float(p.math_mode), float(p.lr), float(p.dt), float(p.friction), float(p.target_speed),
            float(p.optimizer)] + [float(x) for x in p.lane_x]


def unpack_params(v: List[float]) -> PlannerParams:
    return PlannerParams(H=int(v[0]), C=int(v[1]), n_iter=int(v[2]), num_lanes=int(v[3]), other_mode=int(v[4]),
                         extra_inits=bool(v[5]), math_mode=int(v[6]), lr=v[7], dt=v[8], friction=v[9],
                         target_speed=v[10], optimizer=int(v[11]), lane_x=tuple(v[12:]))


@torch.library.custom_op("ocd_b200::solve", mutates_args=())
def solve(world: torch.Tensor, weights: torch.Tensor, weight_idx: Optional[torch.Tensor],
          other_controls: Optional[torch.Tensor], params: List[float]) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """world [C,4,B] f32, weights [K,Bw] f32, weight_idx [B] i32 | None, other_controls [C-1,H,2,Bo] f32 | None
    -> (plan [H,2,B], losses [S,B], best [B] i32): NaivePlanner.generate_plan for B problems."""
    p = unpack_params(params)
    eng = _engine(world)
    Bo = 0 if other_controls is None else other_controls.shape[-1]
    out = eng.solve_soa(p, world.contiguous(), weights.contiguous(), weights.shape[-1],
                        None if weight_idx is None else weight_idx.contiguous(),
                        None if other_controls is None else other_controls.contiguous(), Bo)
    return out["plan"], out["losses"], out["best"]


@solve.register_fake
def _(world, weights, weight_idx, other_controls, params):
    p = unpack_params(params)
    B = world.shape[-1]
    return (world.new_empty((p.H, 2, B)), world.new_empty((p.S, B)), world.new_empty((B,), dtype=torch.int32))


@torch.library.custom_op("ocd_b200::solve_vjp", mutates_args=())
def solve_vjp(world: torch.Tensor, weights: torch.Tensor, weight_idx: Optional[torch.Tensor],
              other_controls: Optional[torch.Tensor], best: torch.Tensor, plan_bar: torch.Tensor,
              params: List[float]) -> Tuple[torch.Tensor, torch.Tensor]:
    """solve's inputs, its `best` [B] i32 and plan_bar [H,2,B] = d loss / d plan -> (weights_bar [K,B]: per problem,
    d loss / d the weight vector problem b planned with; world_bar [C,4,B])."""
    p = unpack_params(params)
    eng = _engine(world)
    Bo = 0 if other_controls is None else other_controls.shape[-1]
    out = eng.solve_vjp_soa(p, world.contiguous(), weights.contiguous(), weights.shape[-1], best.contiguous(),
                            plan_bar.contiguous(), None if weight_idx is None else weight_idx.contiguous(),
                            None if other_controls is None else other_controls.contiguous(), Bo)
    return out["weights_bar"], out["world_bar"]


@solve_vjp.register_fake
def _(world, weights, weight_idx, other_controls, best, plan_bar, params):
    p = unpack_params(params)
    B = world.shape[-1]
    return world.new_empty((p.K, B)), world.new_empty((p.C, 4, B))


@torch.library.custom_op("ocd_b200::solve_implicit_vjp", mutates_args=())
def solve_implicit_vjp(world: torch.Tensor, weights: torch.Tensor, weight_idx: Optional[torch.Tensor],
                       other_controls: Optional[torch.Tensor], plan: torch.Tensor, plan_bar: torch.Tensor,
                       params: List[float]) -> Tuple[torch.Tensor, torch.Tensor]:
    """solve's inputs with L-BFGS params, its plan [H,2,B] and plan_bar [H,2,B] = d loss / d plan -> (weights_bar [K,B]:
    per problem; world_bar [C,4,B]): the implicit-function derivative of the optimum the plan stands for."""
    p = unpack_params(params)
    eng = _engine(world)
    Bo = 0 if other_controls is None else other_controls.shape[-1]
    out = eng.solve_implicit_vjp_soa(p, world.contiguous(), weights.contiguous(), weights.shape[-1], plan.contiguous(),
                                     plan_bar.contiguous(), None if weight_idx is None else weight_idx.contiguous(),
                                     None if other_controls is None else other_controls.contiguous(), Bo)
    return out["weights_bar"], out["world_bar"]


@solve_implicit_vjp.register_fake
def _(world, weights, weight_idx, other_controls, plan, plan_bar, params):
    p = unpack_params(params)
    B = world.shape[-1]
    return world.new_empty((p.K, B)), world.new_empty((p.C, 4, B))


def _solve_setup_context(ctx, inputs, output):
    world, weights, weight_idx, other_controls, params = inputs
    ctx.set_materialize_grads(False)          # an output nobody differentiates arrives as None, not as zeros
    ctx.save_for_backward(world, weights, weight_idx, other_controls, output[2], output[0])
    ctx.params = params


def _solve_backward(ctx, plan_bar, losses_bar, best_bar):
    if losses_bar is not None:
        raise RuntimeError("ocd_b200::solve: the losses are not differentiable (only the plan is: the gradient follows "
                           "the winning start through the SGD iterations); detach them before using them in a loss")
    if ctx.needs_input_grad[3]:
        raise RuntimeError("ocd_b200::solve: gradients with respect to other_controls are not supported; "
                           "pass other_controls without requires_grad")
    world, weights, weight_idx, other_controls, best, plan = ctx.saved_tensors
    if plan_bar is None:
        return None, None, None, None, None
    if unpack_params(ctx.params).optimizer == 1:
        # L-BFGS: the derivative of the optimum the plan stands for (the line search is not differentiated)
        weights_bar, world_bar = torch.ops.ocd_b200.solve_implicit_vjp(world, weights, weight_idx, other_controls,
                                                                       plan, plan_bar.contiguous(), ctx.params)
    else:
        weights_bar, world_bar = torch.ops.ocd_b200.solve_vjp(world, weights, weight_idx, other_controls, best,
                                                              plan_bar.contiguous(), ctx.params)
    Bw, B = weights.shape[-1], world.shape[-1]
    if weight_idx is not None:
        # rows of the problems that share a vector, summed deterministically: index_put_ with accumulate=True sorts by
        # index on CUDA (index_add_ would add with float atomics, in an order that changes from run to run)
        wb = torch.zeros((Bw, weights_bar.shape[0]), dtype=weights_bar.dtype, device=weights_bar.device)
        wb.index_put_((weight_idx.long(),), weights_bar.t(), accumulate=True)
        weights_bar = wb.t()
    elif Bw == 1 and B != 1:
        weights_bar = weights_bar.sum(dim=1, keepdim=True)
    return (world_bar if ctx.needs_input_grad[0] else None, weights_bar if ctx.needs_input_grad[1] else None,
            None, None, None)


solve.register_autograd(_solve_backward, setup_context=_solve_setup_context)


@torch.library.custom_op("ocd_b200::episodes", mutates_args=())
def episodes(robot_init: torch.Tensor, plan_weights: torch.Tensor, weight_idx: Optional[torch.Tensor],
             true_weights: torch.Tensor, unlucky_idx: Optional[torch.Tensor], params: List[float],
             scenario: List[float], T: int) -> torch.Tensor:
    """robot_init [4,B], plan_weights [K,Bw], true_weights [K] -> returns [B]: MPC_ORD's episode loop.
    `scenario` is `pack_scenario(...)`."""
    p = unpack_params(params)
    sc = unpack_scenario(scenario)
    eng = _engine(robot_init)
    out = eng.episodes_soa(p, sc, robot_init.contiguous(), plan_weights.contiguous(), plan_weights.shape[-1],
                           true_weights.contiguous(), int(T),
                           weight_idx=None if weight_idx is None else weight_idx.contiguous(),
                           unlucky_idx=None if unlucky_idx is None else unlucky_idx.contiguous())
    return out["returns"]


@episodes.register_fake
def _(robot_init, plan_weights, weight_idx, true_weights, unlucky_idx, params, scenario, T):
    return robot_init.new_empty((robot_init.shape[-1],))


@torch.library.custom_op("ocd_b200::episodes_trace", mutates_args=())
def episodes_trace(robot_init: torch.Tensor, plan_weights: torch.Tensor, weight_idx: Optional[torch.Tensor],
                   true_weights: torch.Tensor, unlucky_idx: Optional[torch.Tensor], params: List[float],
                   scenario: List[float], T: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """episodes with its per-step trace -> (returns [B], controls [T,2,B], best [T,B] i32, states [T,C,4,B]): the same
    kernel and the same bits as episodes; what episodes_vjp differentiates along."""
    p = unpack_params(params)
    sc = unpack_scenario(scenario)
    eng = _engine(robot_init)
    out = eng.episodes_soa(p, sc, robot_init.contiguous(), plan_weights.contiguous(), plan_weights.shape[-1],
                           true_weights.contiguous(), int(T),
                           weight_idx=None if weight_idx is None else weight_idx.contiguous(),
                           unlucky_idx=None if unlucky_idx is None else unlucky_idx.contiguous(), trace=True)
    return out["returns"], out["controls"], out["best"], out["states"]


@episodes_trace.register_fake
def _(robot_init, plan_weights, weight_idx, true_weights, unlucky_idx, params, scenario, T):
    p = unpack_params(params)
    B = robot_init.shape[-1]
    return (robot_init.new_empty((B,)), robot_init.new_empty((T, 2, B)),
            robot_init.new_empty((T, B), dtype=torch.int32), robot_init.new_empty((T, p.C, 4, B)))


@torch.library.custom_op("ocd_b200::episodes_vjp", mutates_args=())
def episodes_vjp(plan_weights: torch.Tensor, weight_idx: Optional[torch.Tensor], true_weights: torch.Tensor,
                 states: torch.Tensor, best: torch.Tensor, controls: torch.Tensor, returns_bar: torch.Tensor,
                 params: List[float], scenario: List[float], T: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """episodes' inputs, the trace of that run (episodes_trace) and returns_bar [B] = d loss / d returns ->
    (plan_weights_bar [K,B]: per world, d loss / d the weight vector world b planned with; robot_init_bar [4,B];
    true_weights_bar [K,B]: per world)."""
    p = unpack_params(params)
    sc = unpack_scenario(scenario)
    eng = _engine(states)
    out = eng.episodes_vjp_soa(p, sc, plan_weights.contiguous(), plan_weights.shape[-1], true_weights.contiguous(),
                               int(T), states.contiguous(), best.contiguous(), controls.contiguous(),
                               returns_bar.contiguous(), None if weight_idx is None else weight_idx.contiguous())
    return out["plan_weights_bar"], out["robot_init_bar"], out["true_weights_bar"]


@episodes_vjp.register_fake
def _(plan_weights, weight_idx, true_weights, states, best, controls, returns_bar, params, scenario, T):
    p = unpack_params(params)
    B = returns_bar.shape[-1]
    return returns_bar.new_empty((p.K, B)), returns_bar.new_empty((4, B)), returns_bar.new_empty((p.K, B))


@torch.library.custom_op("ocd_b200::episodes_implicit_vjp", mutates_args=())
def episodes_implicit_vjp(plan_weights: torch.Tensor, weight_idx: Optional[torch.Tensor], true_weights: torch.Tensor,
                          states: torch.Tensor, best: torch.Tensor, controls: torch.Tensor, returns_bar: torch.Tensor,
                          params: List[float], scenario: List[float],
                          T: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """episodes_vjp for L-BFGS params: every step's control Jacobian by the implicit function theorem at its plan
    -> (plan_weights_bar [K,B], robot_init_bar [4,B], true_weights_bar [K,B]), per world."""
    p = unpack_params(params)
    sc = unpack_scenario(scenario)
    eng = _engine(states)
    out = eng.episodes_implicit_vjp_soa(p, sc, plan_weights.contiguous(), plan_weights.shape[-1],
                                        true_weights.contiguous(), int(T), states.contiguous(), best.contiguous(),
                                        controls.contiguous(), returns_bar.contiguous(),
                                        None if weight_idx is None else weight_idx.contiguous())
    return out["plan_weights_bar"], out["robot_init_bar"], out["true_weights_bar"]


@episodes_implicit_vjp.register_fake
def _(plan_weights, weight_idx, true_weights, states, best, controls, returns_bar, params, scenario, T):
    p = unpack_params(params)
    B = returns_bar.shape[-1]
    return returns_bar.new_empty((p.K, B)), returns_bar.new_empty((4, B)), returns_bar.new_empty((p.K, B))


def _episodes_setup_context(ctx, inputs, output):
    robot_init, plan_weights, weight_idx, true_weights, unlucky_idx, params, scenario, T = inputs
    ctx.save_for_backward(robot_init, plan_weights, weight_idx, true_weights, unlucky_idx)
    ctx.params, ctx.scenario, ctx.T = params, scenario, T


def _episodes_backward(ctx, returns_bar):
    robot_init, plan_weights, weight_idx, true_weights, unlucky_idx = ctx.saved_tensors
    # the trace of the forward's own run: the same kernel on the same inputs, so the same bits
    _, controls, best, states = torch.ops.ocd_b200.episodes_trace(robot_init, plan_weights, weight_idx, true_weights,
                                                                  unlucky_idx, ctx.params, ctx.scenario, ctx.T)
    # L-BFGS: the implicit-function derivative of every step's optimum (the line search is not differentiated)
    vjp = torch.ops.ocd_b200.episodes_implicit_vjp if unpack_params(ctx.params).optimizer == 1 \
        else torch.ops.ocd_b200.episodes_vjp
    pw_bar, ri_bar, tw_bar = vjp(plan_weights, weight_idx, true_weights, states, best, controls,
                                 returns_bar.contiguous(), ctx.params, ctx.scenario, ctx.T)
    Bw, B = plan_weights.shape[-1], robot_init.shape[-1]
    if weight_idx is not None:
        # rows of the worlds that share a vector, summed deterministically (see _solve_backward)
        wb = torch.zeros((Bw, pw_bar.shape[0]), dtype=pw_bar.dtype, device=pw_bar.device)
        wb.index_put_((weight_idx.long(),), pw_bar.t(), accumulate=True)
        pw_bar = wb.t()
    elif Bw == 1 and B != 1:
        pw_bar = pw_bar.sum(dim=1, keepdim=True)
    return (ri_bar if ctx.needs_input_grad[0] else None, pw_bar if ctx.needs_input_grad[1] else None, None,
            tw_bar.sum(dim=1) if ctx.needs_input_grad[3] else None, None, None, None, None)


episodes.register_autograd(_episodes_backward, setup_context=_episodes_setup_context)


def pack_scenario(sc: Scenario) -> List[float]:
    """Scenario -> flat list: [n, critical_t, teleport(4), then per car: kind, friction, init(4), control(2),
    plan_len, plan(2*plan_len)]."""
    v = [float(len(sc.init_state)), float(sc.critical_t)] + [float(x) for x in sc.teleport_state]
    for j in range(len(sc.init_state)):
        pl = sc.plan[j] if j < len(sc.plan) else ()
        v += [float(sc.kind[j]), float(sc.friction[j])] + [float(x) for x in sc.init_state[j]] + \
             [float(x) for x in sc.control[j]] + [float(len(pl))]
        for u in pl:
            v += [float(u[0]), float(u[1])]
    return v


def unpack_scenario(v: List[float]) -> Scenario:
    n, crit, tele = int(v[0]), int(v[1]), tuple(v[2:6])
    i = 6
    kind, fric, init, ctrl, plans = [], [], [], [], []
    for _ in range(n):
        kind.append(int(v[i])); fric.append(v[i + 1]); init.append(list(v[i + 2:i + 6])); ctrl.append(list(v[i + 6:i + 8]))
        m = int(v[i + 8])
        plans.append([[v[i + 9 + 2 * q], v[i + 10 + 2 * q]] for q in range(m)])
        i += 9 + 2 * m
    return Scenario(init_state=init, kind=kind, friction=fric, control=ctrl, plan=plans, critical_t=crit,
                    teleport_state=tele)
