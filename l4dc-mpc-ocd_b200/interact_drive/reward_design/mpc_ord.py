"""MPC_ORD and the finite_horizon scenario: mirror of interact_drive/reward_design/mpc_ord.py of the
reference (MPC_ORD :15-158, finite_horizon_env :162-207).

The reference evaluates a weight vector by resetting a Python world and stepping it `designer_horizon`
times for every initial state and sample, one full MPC solve per step.  Here a whole evaluation -- all
initial states x samples, and in `eval_weights_batch` all candidates of a CMA-ES generation too -- is
one launch of the episode kernel (`ocd_episode_batch`); the Python world is only compiled into the
POD description the kernel needs."""
from __future__ import annotations

import pickle
import sys
import time
from typing import Optional, Sequence

import math

import numpy as np
import scipy.stats

from ... import cmaes as _cma
from ... import parallel as _par
from ...batched import compile_world, unlucky_sequence
from ...experiments.merging import ThreeLaneCarWorld, ThreeLaneTestCar
from ...runtime import as_f32, get_engine
from ..car import FixedVelocityCar


class list2(list):
    """A list that can carry attributes (`history.seed`), pickled under the reference's module path so
    that the reference's loaders (experiments/generalization_data.py:18) read our histories."""

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)


list2.__module__ = "interact_drive.reward_design.mpc_ord"


def _truncnorm_sample(mean, std, rang):
    a, b = (rang[0] - mean) / std, (rang[1] - mean) / std
    return np.squeeze(scipy.stats.truncnorm.rvs(a, b) * std + mean)


def sample_init_state(env_seed, x, y, speed):
    """Robot initial state: three truncated normals drawn under np.random.seed(env_seed), heading pi/2
    (reference mpc_ord.py:171-181; scipy-version dependent, so parity tests pass states explicitly)."""
    np.random.seed(seed=env_seed)
    return np.array([_truncnorm_sample(*x), _truncnorm_sample(*y), _truncnorm_sample(*speed), np.pi / 2])


def _unit_rows(W: np.ndarray) -> np.ndarray:
    """w / np.linalg.norm(w) for every row of W [n, K] (float64): np.linalg.norm of a real vector is sqrt(x.dot(x)),
    and np.vecdot runs that same BLAS dot over each row, so the quotients are the per-row ones bit for bit -- in one
    call instead of n."""
    return W / np.sqrt(np.vecdot(W, W))[:, None]


def _planning_weight_rows(W: np.ndarray) -> np.ndarray:
    """MPC_ORD._planning_weights for every row of W [n, K]: three normalisations in float64, then the cast."""
    for _ in range(3):
        W = _unit_rows(W)
    return W.astype(np.float32)


def _planning_weights_vjp(w: np.ndarray, g: np.ndarray) -> np.ndarray:
    """The transposed Jacobian of MPC_ORD._planning_weights's three float64 normalisations at the raw vector w [K],
    applied to g = d f / d (planning weights): -> d f / d w (float64; the final cast to float32 counts as the identity).
    The normalisation x -> x / |x| has the Jacobian (I - u u^T) / |x|, u = x / |x|."""
    xs = [np.asarray(w, dtype=np.float64)]
    for _ in range(2):
        xs.append(xs[-1] / math.sqrt(float(xs[-1].dot(xs[-1]))))
    g = np.asarray(g, dtype=np.float64)
    for x in reversed(xs):
        n = math.sqrt(float(x.dot(x)))
        u = x / n
        g = (g - u * float(u.dot(g))) / n
    return g


def _launch_sharded(eng, ord_, W, robot, widx, unlucky):
    """One process per GPU: this rank runs its contiguous shard of the episodes, then the per-episode rows -- return
    and final world state -- are all-gathered (the path's only exchange step), so every rank holds the same data and
    leaves the same Python-object state behind as a single-GPU run.  -> (returns [B], final world [C, 4] of the
    last episode), host arrays."""
    p, B = ord_.program.params, robot.shape[0]

    def run(idx):
        o = eng.episodes(p, ord_.program.scenario, robot[idx], W, as_f32(ord_.designer_weights), ord_.designer_horizon,
                         weight_idx=widx[idx], unlucky_idx=None if unlucky is None else unlucky[idx], final_world=True)
        import torch
        return torch.cat([o["returns"][:, None], o["final_world"].reshape(len(idx), -1)], dim=1)

    rows = _par.sharded_rows(run, B).cpu().numpy()
    return np.ascontiguousarray(rows[:, 0]), rows[-1, 1:].reshape(p.C, 4)


def _run_signature(r: "MPC_ORD") -> tuple:
    """What two MPC_ORDs must share to be evaluated in one launch (the compiled structs are kept per object)."""
    sig = getattr(r, "_lockstep_sig", None)
    if sig is None:
        sig = r._lockstep_sig = (bytes(r.program.params.c_struct()), bytes(r.program.scenario.c_struct()))
    return sig + (r.designer_horizon, r.num_samples, as_f32(r.designer_weights).tobytes())


def _candidate_rows(wl, K: int) -> np.ndarray:
    """One run's candidates as a float64 [n, K] array (rows may come as [K] or [1, K], like the reference passes them)."""
    if isinstance(wl, np.ndarray) and wl.ndim == 2 and wl.shape[1] == K:
        return np.asarray(wl, dtype=np.float64)
    if len(wl) == 0:
        return np.zeros((0, K))
    rows = [np.asarray(w, dtype=np.float64) for w in wl]
    return np.stack([w[0] if w.ndim == 2 else w for w in rows])


def eval_weights_lockstep(runs: Sequence["MPC_ORD"], weight_lists: Sequence[Sequence],
                          session: Optional[dict] = None) -> list:
    """`eval_weights_batch` for several independent MPC_ORDs in ONE launch: run r evaluates weight_lists[r] (possibly
    empty) on ITS initial states.  The reference runs such optimisations in separate worker processes
    (`Pool(len(init_states_groups))`, experiments/run_mpc_ord.py:83-90); here their generations share a kernel launch
    -- sharded over the ranks when a process group is up -- and every run's history advances exactly as if it had
    been evaluated alone (each episode's result does not depend on what else is in the batch).  The host side of a
    generation is vectorised over the runs too -- one normalisation of all candidates, one launch through the host
    context with the episode layout kept between generations -- because with many runs it, not the launch, is what a
    generation costs.
    `session`: a dict the caller keeps across the calls of ONE optimisation (optimize_cmaes_lockstep does): the runs
    are checked against each other once, and the state a serial evaluation leaves in the Python objects (last weights,
    last initial state, final world) is parked in it instead of being written after every generation --
    `finish_lockstep_session` writes it at the end.  Without it every call checks and writes.
    -> list of -totals arrays, one per run."""
    runs = list(runs)
    ref = runs[0]
    if session is None or not session.get("checked"):
        sig = _run_signature(ref)
        for r in runs[1:]:
            if _run_signature(r) != sig:
                raise ValueError("eval_weights_lockstep: the runs must share scenario, planner and designer weights")
        if session is not None:
            session["checked"] = True
    K = ref.program.params.K
    lists = [_candidate_rows(wl, K) for wl in weight_lists]
    active = [i for i, wl in enumerate(lists) if len(wl)]
    if not active:
        return [np.zeros(0) for _ in runs]
    raw = np.concatenate([lists[i] for i in active])                   # every candidate of every active run
    W = _planning_weight_rows(raw)                                     # what the planner gets  [sum nc, K] float32
    unit = _unit_rows(raw)                                             # what the history records (reference :120)
    # the episode layout of a run -- its initial states tiled over its candidates -- is kept for the session (the
    # initial states do not change inside one optimisation); the replanning world's vanishing cars are drawn per call
    kept = None if session is None else session.setdefault("layouts", {})
    layouts = []
    for i in active:
        nc = len(lists[i])
        l = None if kept is None else kept.get((i, nc))
        if l is None:
            l = runs[i]._episode_layout(nc, with_unlucky=False)
            if kept is not None:
                kept[(i, nc)] = l
        layouts.append(l)
    counts = np.array([len(lists[i]) for i in active])
    offs = np.concatenate([[0], np.cumsum(counts)])
    # the flat episode batch: kept between generations while the same runs evaluate as many candidates on the same
    # initial states (the arrays of a layout are themselves kept per run, so identity is the test)
    cache = getattr(ref, "_lockstep_cache", None)
    key = tuple((i, id(l["robot"]), id(l["widx"])) for i, l in zip(active, layouts))
    if cache is None or cache["key"] != key:
        robot = np.concatenate([l["robot"] for l in layouts])
        widx = np.concatenate([l["widx"] + o for l, o in zip(layouts, offs)]).astype(np.int32)
        cache = ref._lockstep_cache = dict(key=key, robot=robot, widx=widx, ri=np.ascontiguousarray(robot.T),
                                           keep=[(l["robot"], l["widx"]) for l in layouts],      # pins the ids
                                           structs=(ref.program.params.c_struct(), ref.program.scenario.c_struct()))
    robot, widx = cache["robot"], cache["widx"]
    unlucky = None
    if ref.program.replanning:
        # the reference resets the world once per (candidate, init, sample), serially, and every reset toggles the
        # vanishing car (reference :87-89, replanning_world.py:19-27): each run's sequence runs over all ITS resets
        unlucky = np.concatenate([unlucky_sequence(runs[i].world, l["robot"].shape[0])
                                  for i, l in zip(active, layouts)]).astype(np.int32)
    p, sc = ref.program.params, ref.program.scenario
    tw = as_f32(ref.designer_weights)
    B = robot.shape[0]
    if _par.world()[1] > 1:
        import torch
        eng = get_engine(ref._device)

        def run(idx):
            o = eng.episodes(p, sc, robot[idx], W, tw, ref.designer_horizon, weight_idx=widx[idx],
                             unlucky_idx=None if unlucky is None else unlucky[idx], final_world=True)
            return torch.cat([o["returns"][:, None], o["final_world"].reshape(len(idx), -1)], dim=1)

        rows = _par.sharded_rows(run, B).cpu().numpy()
        ret, fw = np.ascontiguousarray(rows[:, 0]), rows[:, 1:].reshape(B, p.C, 4)
    else:
        from ...runtime import get_host_context
        ret, fw = get_host_context(ref._device).episodes_soa(
            p, sc, cache["ri"], np.ascontiguousarray(W.T), tw, ref.designer_horizon, weight_idx=widx,
            unlucky_idx=unlucky, final_world=True, structs=cache["structs"])
        fw = np.moveaxis(fw, -1, 0)                                      # [C, 4, B] -> [B, C, 4]
    ref.kernel_launches += 1
    # per-candidate totals: when every run has the same (candidates, inits, samples) -- lock step on equally large init
    # groups -- one reduction for all of them (rows of ni*ns contiguous returns: the sum _record takes per run)
    shape0 = layouts[0]["shape"]
    totals_all = None
    if all(l["shape"] == shape0 for l in layouts):
        totals_all = ret.reshape(-1, shape0[1] * shape0[2]).sum(axis=1, dtype=np.float64) / ref.num_samples
    out, at = [np.zeros(0) for _ in runs], 0
    state = None if session is None else session.setdefault("state", {})
    for j, i in enumerate(active):
        l = layouts[j]
        n = l["robot"].shape[0]
        lo, hi = offs[j], offs[j + 1]
        if state is None:
            runs[i]._after_episodes(dict(W=W[lo:hi], I=l["I"]), fw[at + n - 1])
        else:
            state[i] = (W[hi - 1], l["I"], fw[at + n - 1])
        out[i] = runs[i]._record(None, None if totals_all is not None else ret[at:at + n].reshape(l["shape"]),
                                 unit[lo:hi], None if totals_all is None else totals_all[lo:hi])
        at += n
    return out


def finish_lockstep_session(runs: Sequence["MPC_ORD"], session: dict) -> None:
    """Write the object state eval_weights_lockstep parked in `session`: every run is left as its last evaluation
    would have left it."""
    runs = list(runs)
    for i, (w_last, I, fw) in session.pop("state", {}).items():
        runs[i]._after_episodes(dict(W=w_last[None].copy(), I=I), fw.copy())


def optimize_cmaes_lockstep(runs: Sequence["MPC_ORD"], seeds: Sequence[int], sigma0=0.1, shard_runs: bool = False,
                            stats: Optional[dict] = None, **stop) -> list:
    """R independent `optimize_cmaes` runs (reference :33-45, one worker process each in the reference) advanced in
    lock step: generation g of every run that is still going is ONE episode launch.  Run r uses seeds[r]; its
    candidates, history and result are those of `runs[r].optimize_cmaes(seed=seeds[r], ...)` run alone.
    With several ranks the episodes of every generation are sharded and all-gathered (every rank keeps all runs'
    books); `shard_runs=True` spreads the RUNS instead -- rank k optimises runs k, k + N, ... on its own GPU with no
    collective, which is how many runs scale end to end (a generation's cost is mostly its Python bookkeeping) -- and
    exchanges histories, results and object state once at the end, so every rank still finishes with all of them
    (`stats`, when given, receives the wall-clock seconds of the two phases: "optimise_s", "exchange_s").
    -> list of best weight vectors."""
    runs = list(runs)
    assert len(seeds) == len(runs)
    rank, ws = _par.group()
    if shard_runs and ws > 1:
        mine = list(range(rank, len(runs), ws))
        t0 = time.perf_counter()
        with _par.local_only():
            xs = optimize_cmaes_lockstep([runs[i] for i in mine], [seeds[i] for i in mine], sigma0, **stop) if mine else []
        t1 = time.perf_counter()
        packed = _par.all_gather_objects([(i, x, runs[i]._export_state()) for i, x in zip(mine, xs)])
        out = [None] * len(runs)
        for part in packed:
            for i, x, state in part:
                out[i] = x
                if i not in mine:
                    runs[i]._import_state(state)
        if stats is not None:
            stats.update(optimise_s=t1 - t0, exchange_s=time.perf_counter() - t1)
        return out
    for r, seed in zip(runs, seeds):
        assert seed != 0
        assert not r.done
        r.history.seed = seed
        r.should_save_history = True
    session = {}
    t0 = time.perf_counter()
    try:
        eval_weights_lockstep(runs, [[r.designer_weights] for r in runs], session)
        res = _cma.fmin2_lockstep(lambda pops: eval_weights_lockstep(runs, pops, session),
                                  [list(r.designer_weights) for r in runs], sigma0,
                                  [dict(seed=seed, **stop) for seed in seeds])
    finally:
        finish_lockstep_session(runs, session)
    if stats is not None:
        stats.update(optimise_s=time.perf_counter() - t0, exchange_s=0.0)
    for r in runs:
        r.should_save_history = False
        r.done = True
    return [x for x, _ in res]


class MPC_ORD:
    """Evaluates / optimises surrogate reward weights for a planning car by the TRUE-weight return of
    the receding-horizon episodes it produces."""

    def __init__(self, world, car, init_car_states, designer_horizon, save_path=None, num_samples=1, *,
                 verbose: bool = True, device: Optional[int] = None):
        self.world, self.car = world, car
        self.designer_horizon = designer_horizon
        self.init_car_states = init_car_states
        self.save_path = save_path
        w = np.asarray(car.weights)
        self.designer_weights = w / np.linalg.norm(w)
        self.weight_dim = len(w)
        # the history is kept as per-evaluation blocks (weights [n, K], totals [n]) and turned into the reference's list
        # of tuples when someone looks (`history`): an optimisation appends thousands of entries nobody reads until
        # the end, and with many runs in lock step the list bookkeeping was a fifth of a generation's host time
        self._history = list2()
        self._history_blocks = []
        self._history_listed = 0        # blocks already in the list
        self.iter = 0
        self.should_save_history = False
        self.done = False
        self.num_samples = num_samples
        self.verbose = verbose
        self._device = device
        self.program = compile_world(world, car)
        self.kernel_launches = 0
        self._dev_cache = {}
        self._batch_cache = None

    # -- the batched core ------------------------------------------------------------------------------
    @staticmethod
    def _planning_weights(weights) -> np.ndarray:
        """What the planner ends up with: normalised in eval_weights, again in eval_weights_for_init and
        again in the car's setter, in float64, then cast (reference :120, :71, linear_reward_car.py:47)."""
        w = np.asarray(weights, dtype=np.float64)
        if w.ndim == 2:
            w = w[0]
        for _ in range(3):
            w = w / math.sqrt(float(w.dot(w)))       # np.linalg.norm of a real vector: sqrt(x.dot(x)), without the call overhead
        return w.astype(np.float32)

    def _episode_batch(self, weight_matrix, inits: Optional[Sequence] = None) -> dict:
        """The flat episode batch of `weight_matrix` [n_cand, K] (raw candidates) x inits [n_init, 4] x num_samples:
        planning weights W [nc, K], robot states [nc*ni*ns, 4], the candidate of every episode and -- replanning world --
        the car that vanishes in it.  Advances the world's own reset toggle like the serial loops would.  Everything
        that depends only on the initial states and the candidate count is kept from one call to the next (the CMA-ES
        loop calls this once per generation with the same states)."""
        Wm = np.atleast_2d(np.asarray(weight_matrix, dtype=np.float64))
        if Wm.ndim == 3:                                     # rows given as [1, K] (the reference passes such weights around)
            Wm = Wm[:, 0, :]
        return dict(W=_planning_weight_rows(Wm), **self._episode_layout(Wm.shape[0], inits))

    def _episode_layout(self, nc: int, inits: Optional[Sequence] = None, with_unlucky: bool = True) -> dict:
        """Everything of `_episode_batch` but the weights, for nc candidates (with_unlucky=False: without drawing the
        replanning world's vanishing cars, which advances the world's toggle -- the caller does that itself)."""
        inits = self.init_car_states if inits is None else inits
        src = np.asarray(inits, dtype=np.float64)
        ns = self.num_samples
        c = self._batch_cache
        if c is None or c["nc"] != nc or c["ns"] != ns or c["src"].shape != src.shape or not np.array_equal(c["src"], src):
            I = np.stack([as_f32(s, (4,)) for s in inits])
            ni = I.shape[0]
            c = dict(nc=nc, ns=ns, src=src.copy(), I=I, robot=np.repeat(np.tile(I, (nc, 1)), ns, axis=0),   # [nc*ni*ns, 4]
                     widx=np.repeat(np.arange(nc, dtype=np.int32), ni * ns))
            self._batch_cache = c
        I, robot, widx = c["I"], c["robot"], c["widx"]
        ni = I.shape[0]
        unlucky = None
        if self.program.replanning and with_unlucky:
            # the reference resets the world once per (candidate, init, sample), serially, and every reset toggles the
            # vanishing car (reference :87-89, replanning_world.py:19-27): the sequence runs over all nc*ni*ns resets
            unlucky = np.asarray(unlucky_sequence(self.world, nc * ni * ns), np.int32)
        return dict(I=I, robot=robot, widx=widx, unlucky=unlucky, shape=(nc, ni, ns))

    @property
    def history(self) -> list2:
        """The reference's history: a list of (normalised weights, -objective) tuples, `history.seed` beside it; entries
        recorded (or received from another rank) since the last look are added now."""
        if self._history_listed < len(self._history_blocks):
            for W, v in self._history_blocks[self._history_listed:]:
                self._history.extend(zip(W, v))
            self._history_listed = len(self._history_blocks)
        return self._history

    @history.setter
    def history(self, value) -> None:
        self._history, self._history_blocks, self._history_listed = value, [], 0

    def _history_arrays(self):
        """The history as (weights [n, K], totals [n]): the blocks, when they still describe the list (nobody appended to
        or cut the list behind its back), else read off the list."""
        listed = sum(len(v) for _, v in self._history_blocks[:self._history_listed])
        if listed == len(self._history):
            if not self._history_blocks:
                return np.zeros((0, self.weight_dim)), np.zeros(0)
            return (np.concatenate([W for W, _ in self._history_blocks]), np.concatenate([v for _, v in self._history_blocks]))
        h = self.history
        return (np.stack([np.asarray(w, dtype=np.float64) for w, _ in h]), np.array([v for _, v in h], dtype=np.float64))

    def _export_state(self) -> dict:
        """What an optimisation leaves in this object (for a rank that did not run it): history, counters, the
        planner's last weights / initial state, the world's final state and the replanning toggle."""
        # the history as two arrays, not thousands of small ones: building, pickling and rebuilding the list is what the
        # exchange would cost otherwise
        return dict(history=self._history_arrays(), seed=getattr(self._history, "seed", None), iter=self.iter, done=self.done,
                    launches=self.kernel_launches, weights=np.asarray(self.car.weights), init=np.asarray(self.car.init_state),
                    states=[np.asarray(c.state) for c in self.world.cars],
                    unlucky=getattr(self.world, "unlucky_car_idx", None))

    def _import_state(self, st: dict) -> None:
        del self._history[:]
        self._history_blocks, self._history_listed = [st["history"]], 0      # list entries are made on first access
        if st["seed"] is not None:
            self._history.seed = st["seed"]
        self.iter, self.done, self.kernel_launches = st["iter"], st["done"], st["launches"]
        self.car.weights_f32 = as_f32(st["weights"])
        self.car.init_state = st["init"]
        for c, s in zip(self.world.cars, st["states"]):
            c.state = s
        if st["unlucky"] is not None:
            self.world.unlucky_car_idx = st["unlucky"]

    def _after_episodes(self, batch: dict, final_world: np.ndarray) -> None:
        """Leave the Python objects the way a serial evaluation would: last weights, last init, final state."""
        self.car.weights = batch["W"][-1]
        self.car.init_state = batch["I"][-1]
        for c, st in zip(self.world.cars, final_world):
            c.state = st

    def episode_returns(self, weight_matrix, inits: Optional[Sequence] = None, trace: bool = False):
        """weight_matrix [n_cand, K] (raw candidates) x inits [n_init, 4] x num_samples ->
        returns [n_cand, n_init, num_samples] of sum_t true_w . features(past_state_t), one launch.
        With trace=True also the per-step controls/states of every episode (host arrays)."""
        batch = self._episode_batch(weight_matrix, inits)
        W, robot, widx, unlucky = batch["W"], batch["robot"], batch["widx"], batch["unlucky"]
        eng = get_engine(self._device)
        rank, ws = _par.world()
        out = None
        if ws > 1 and not trace:
            ret_flat, final = _launch_sharded(eng, self, W, robot, widx, unlucky)
        elif not trace:
            # the CMA-ES hot loop: everything but the candidates is the same from one generation to the next, so
            # the device copies of the initial states / indices are kept, only W goes up and ONE buffer (returns +
            # final worlds) comes back
            ret_flat, final = self._episode_returns_cached(eng, W, robot, widx, unlucky)
        else:
            out = eng.episodes(self.program.params, self.program.scenario, robot, W, as_f32(self.designer_weights),
                               self.designer_horizon, weight_idx=widx, unlucky_idx=unlucky, trace=trace,
                               final_world=True)
            ret_flat = out["returns"].cpu().numpy()
            final = out["final_world"].cpu().numpy()[-1]
        self.kernel_launches += 1
        self._after_episodes(batch, final)
        ret = ret_flat.reshape(batch["shape"])
        if trace:
            return ret, {k: out[k].cpu().numpy() for k in ("controls", "best", "states")}
        return ret

    # -- reference API -----------------------------------------------------------------------------------
    def _episode_returns_cached(self, eng, W, robot, widx, unlucky):
        """-> (returns [B] host, final world [C, 4] of the last episode); see episode_returns.
        The CMA-ES hot loop: numpy in, numpy out through `ocd_episode_batch_host`, whose context keeps the staging
        buffers and replays ONE captured CUDA graph (copy-in, episode kernel, copy-out) per generation; the SoA
        transposes of everything but the candidates and the two C structs are cached here."""
        from ...runtime import get_host_context
        p, sc = self.program.params, self.program.scenario
        B = robot.shape[0]
        key = (robot.tobytes(), widx.tobytes(), None if unlucky is None else unlucky.tobytes(),
               as_f32(self.designer_weights).tobytes())
        c = self._dev_cache.get(key)
        if c is None:
            if len(self._dev_cache) >= 8:
                self._dev_cache.clear()
            c = dict(ri=np.ascontiguousarray(robot.T), idx=np.ascontiguousarray(widx, np.int32),
                     tw=as_f32(self.designer_weights), ul=None if unlucky is None else np.ascontiguousarray(unlucky, np.int32),
                     structs=(p.c_struct(), sc.c_struct()))
            self._dev_cache[key] = c
        ret, fw = get_host_context(self._device).episodes_soa(
            p, sc, c["ri"], np.ascontiguousarray(W.T), c["tw"], self.designer_horizon, weight_idx=c["idx"],
            unlucky_idx=c["ul"], final_world=True, structs=c["structs"])
        return ret, fw[:, :, -1]

    def eval_weights_for_init(self, init, weights, render=False, heatmap_show=False):
        """Return of `weights` from one initial state, summed over the samples (reference :67-106)."""
        if render:
            raise NotImplementedError("rendering is outside the batched MPC engine's scope")
        r = self.episode_returns([weights], [init], trace=self.car.debug)
        if self.car.debug:
            r, tr = r
            ctl, st = tr["controls"][-1], tr["states"][-1]          # the last sample, like a serial run leaves
            for j, c in enumerate(self.world.cars):
                c.past_traj = [(st[t, j].copy(), ctl[t].copy() if j == 0 else None) for t in range(st.shape[0])]
        total = np.float32(r[0, 0].sum(dtype=np.float32))
        if self.verbose:
            print('init', init, 'weights', self.car.weights, '\tgave return:', total, 'time', time.time())
        return total

    def eval_weights(self, weights, gif=None, heatmap_show=False):
        """-> MINUS the return of `weights` summed over the initial states and averaged over samples
        (reference :109-151): the callable CMA-ES minimises."""
        if gif:
            raise NotImplementedError("gif rendering is outside the batched MPC engine's scope")
        return float(self.eval_weights_batch([weights])[0])

    def eval_weights_grad(self, weights):
        """-> (objective, grad): the objective is eval_weights(weights) bit for bit -- the same episode kernel on the same
        batch, launched through the traced device path -- and grad its gradient with respect to the raw candidate
        `weights` [K] (float64): the episodes' reverse pass (``ocd_episode_vjp_batch``) summed over the initial states
        and samples, divided by the samples, through the three normalisations of _planning_weights.  History, iteration
        counter and the replanning world's reset toggle advance exactly as in eval_weights, so the two can be mixed in
        one optimisation."""
        import torch
        w = np.asarray(weights, dtype=np.float64)
        w = w[0] if w.ndim == 2 else w
        batch = self._episode_batch([w])
        W, robot, widx, unlucky = batch["W"], batch["robot"], batch["widx"], batch["unlucky"]
        p, sc, T = self.program.params, self.program.scenario, self.designer_horizon
        eng = get_engine(self._device)
        dev = eng.device
        ri = torch.as_tensor(np.ascontiguousarray(robot.T), device=dev)
        wp = torch.as_tensor(np.ascontiguousarray(W.T), device=dev)
        tw = torch.as_tensor(as_f32(self.designer_weights), device=dev)
        idx = torch.as_tensor(widx, device=dev)
        ul = None if unlucky is None else torch.as_tensor(unlucky, device=dev)
        out = eng.episodes_soa(p, sc, ri, wp, 1, tw, T, weight_idx=idx, unlucky_idx=ul, trace=True, final_world=True)
        vjp = eng.episodes_vjp_soa(p, sc, wp, 1, tw, T, out["states"], out["best"], out["controls"],
                                   torch.ones_like(out["returns"]), weight_idx=idx, robot_init_bar=False,
                                   true_weights_bar=False)
        ret = out["returns"].cpu().numpy()
        self.kernel_launches += 1
        self._after_episodes(batch, out["final_world"][:, :, -1].cpu().numpy())
        objective = float(self._record([w], ret.reshape(batch["shape"]))[0])
        # objective = -sum(returns) / num_samples
        g_plan = -vjp["plan_weights_bar"].cpu().numpy().astype(np.float64).sum(axis=1) / self.num_samples
        return objective, _planning_weights_vjp(w, g_plan)

    def eval_weights_batch(self, weight_matrix) -> np.ndarray:
        """eval_weights for every row of weight_matrix in ONE launch; history and iteration counter
        advance exactly as if the rows had been evaluated one after the other."""
        W = [np.asarray(w, dtype=np.float64) for w in weight_matrix]
        W = [w[0] if w.ndim == 2 else w for w in W]
        return self._record(W, self.episode_returns(W))               # [nc, ni, ns]

    def _record(self, W, ret, unit=None, totals=None) -> np.ndarray:
        """History / iteration bookkeeping of eval_weights (reference :128-151) for the candidates W with episode
        returns ret [nc, ni, ns].  `unit`: the rows w / np.linalg.norm(w) (reference :120), `totals`: the per-candidate
        sums over (ni, ns) divided by the samples, when the caller has them already.  -> -totals."""
        if totals is None:
            totals = ret.sum(axis=(1, 2), dtype=np.float64) / self.num_samples
        if unit is None:
            unit = _unit_rows(np.asarray(W, dtype=np.float64).reshape(len(totals), -1))
        if self.verbose:
            for k, (wn, total) in enumerate(zip(unit, totals)):
                print('ITERATION', self.iter + k)
                print('eval', wn)
                print('eval reward for weights:', total, '\n\n')
        # rows of a fresh array (nothing else refers to them); `history` turns the block into list entries on demand
        self._history_blocks.append((unit.copy(), np.asarray(totals, dtype=np.float64)))
        self.iter += len(totals)
        if self.should_save_history and self.save_path is not None:
            self.save_history()
        return -totals

    def optimize_cmaes(self, seed=1, sigma0=0.1, **stop):
        """CMA-ES over the weights starting from the designer's (reference :33-45); every generation is
        one launch.  `stop` forwards maxfevals / maxiter / tolfun / tolx."""
        self.history.seed = seed
        assert seed != 0
        assert not self.done
        self.should_save_history = True
        self.eval_weights(self.designer_weights)
        x, es = _cma.fmin2(self.eval_weights, list(self.designer_weights), sigma0, dict(seed=seed, **stop),
                           batch_objective=self.eval_weights_batch)
        self.should_save_history = False
        self.done = True
        return x

    def optimize_random_search(self, n_iter=1000, seed=1, chunk=256):
        """Uniform random search in [-1, 1]^K (reference :47-65), `chunk` candidates per launch."""
        self.history.seed = seed
        assert not self.done
        self.should_save_history = True
        if self.verbose:
            print("\n\nSTARTING RANDOM SEARCH")
        self.iter = 0
        self.eval_weights(self.designer_weights)
        np.random.seed(seed)
        cands = [np.random.rand(*self.designer_weights.shape) * 2 - 1 for _ in range(n_iter)]
        for i in range(0, n_iter, chunk):
            self.eval_weights_batch(cands[i:i + chunk])
        self.should_save_history = False
        self.done = True
        return max(self.history, key=lambda a: a[1])

    def save_history(self):
        assert self.save_path is not None
        # list2 pickles as interact_drive.reward_design.mpc_ord.list2 (the reference's path)
        pkg = __name__.rsplit(".interact_drive.", 1)[0]
        for alias in ("interact_drive", "interact_drive.reward_design", "interact_drive.reward_design.mpc_ord"):
            sys.modules.setdefault(alias, sys.modules[pkg + "." + alias])
        if getattr(sys.modules["interact_drive.reward_design.mpc_ord"], "list2", None) is not list2:
            raise RuntimeError("another interact_drive.reward_design.mpc_ord is imported; cannot pickle history")
        with open(self.save_path, 'wb') as file:
            pickle.dump(self.history, file)
        if self.verbose:
            print('Wrote results so far to', self.save_path)


def finite_horizon_env(horizon=5, env_seeds=[1], debug=True, extra_inits=False):
    """The finite-horizon scenario (reference mpc_ord.py:162-207): a three-lane road, the planning car
    behind a slower FixedVelocityCar in its lane.  -> (car, world, init_states)."""
    init_states = [sample_init_state(s, (0, 0.04, (-0.1, 0.1)), (-0.9, 0.02, (-0.95, -0.85)), (0.8, 0.03, (0.7, 0.9)))
                   for s in env_seeds]
    world = ThreeLaneCarWorld(visualizer_args=dict(name="Switch Lanes"))
    planner_args = dict(n_iter=200 if horizon == 6 else 100, extra_inits=extra_inits)
    our_car = ThreeLaneTestCar(world, init_state=init_states[0], horizon=horizon,
                               weights=np.array([-5, 0., 0., 0., -6., -50, -50]), debug=debug,
                               planner_args=planner_args)
    other_car = FixedVelocityCar(world, np.array([0, -0.6, 0.5, np.pi / 2]), color="gray", opacity=0.8, debug=debug)
    world.add_cars([our_car, other_car])
    world.reset()
    return our_car, world, init_states
