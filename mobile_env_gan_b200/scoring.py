"""Layout scoring (SURVEY.md 8(f)-3): the fork searches BS layouts by running an episode per
random layout and ranking them with ``qoeValue`` (mobile_env/chooseBaseStation.ipynb cell 5):

    score = w1 * mean(qoe) - w2 * var(qoe) - w3 * P(qoe < low_qoe_threshold)

over all two-decimal per-UE QoE values of the epoch (base.py:269).  With one env per layout the
whole search is a batch: ``LayoutScorer`` accumulates the statistics on the device after every
step (``mbe_accumulate_qoe``) and ranks the envs without any file round trip.

With ``num_trajectories`` = M > 1 (DESIGN.md section 10) a layout is scored over M UE trajectories:
layout l occupies the env rows l*M .. l*M + M-1, replica m follows trajectory m, and the score is
``qoeValue`` over all QoE values of the M episodes, so every layout sees the same M trajectories."""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch

from . import _lib


def check_layouts(plan, bs_xy, nbs, L):
    """Host check of L layouts for an env with random per-env layouts: shapes bs_xy [L, B, 2] /
    nbs [L], counts in the scenario's ``bs_random`` range, live BSs on the map.  Returns int16 / int32
    numpy copies with the slots at or beyond nbs set to (0, 0)."""
    B = plan.num_bs
    nmin, nmax = plan.bs_random[0], min(plan.bs_random[1], B)
    xy = np.asarray(torch.as_tensor(bs_xy).cpu(), dtype=np.int64)
    n = np.asarray(torch.as_tensor(nbs).cpu(), dtype=np.int64)
    if xy.shape != (L, B, 2) or n.shape != (L,):
        raise ValueError(f"a population must be bs_xy [{L}, {B}, 2] and nbs [{L}], got "
                         f"{tuple(xy.shape)} and {tuple(n.shape)}")
    if n.min() < nmin or n.max() > nmax:
        raise ValueError(f"nbs must lie in [{nmin}, {nmax}]")
    xm, ym = math.ceil(plan.width) - 1, math.ceil(plan.height) - 1
    live = np.arange(B)[None, :] < n[:, None]
    x, y = xy[..., 0][live], xy[..., 1][live]
    if x.size and (x.min() < 0 or x.max() > xm or y.min() < 0 or y.max() > ym):
        raise ValueError(f"BS coordinates must lie in [0, {xm}] x [0, {ym}]")
    return np.where(live[..., None], xy, 0).astype(np.int16), n.astype(np.int32)


class LayoutScorer:
    """Scores the env's BS layouts: one per env, or with ``num_trajectories`` = M > 1 one per group of
    M env rows (``num_layouts`` = num_envs / M), pooled over the M trajectories."""

    def __init__(self, env, low_qoe_threshold: float = 0.0, weights=(1.0, 0.1, 10.0)):
        self.env, self.threshold, self.weights = env, float(low_qoe_threshold), weights
        self.M = env.plan.num_trajectories
        self.num_layouts = env.num_envs // self.M
        self.acc = torch.zeros(env.num_envs, 4, dtype=torch.float32, device=env.device)

    def reset(self):
        self.acc.zero_()

    def update(self):
        """Call after every ``env.step``."""
        env = self.env
        _lib.check(env._lib.mbe_accumulate_qoe(env._handle, C.c_void_p(self.acc.data_ptr()),
                                               C.c_float(self.threshold), env._stream()))

    def run_episode(self, steps: int = None, record=()):
        """One whole episode through ``mbe_rollout`` with the statistics accumulated inside the
        kernel (one launch for the fork's own scenario) instead of ``step`` + ``update`` per step."""
        env = self.env
        return env.rollout(env.plan.ep_time if steps is None else steps, qoe_acc=self.acc,
                           threshold=self.threshold, record=record)

    def pooled(self):
        """The four accumulators per layout, f32 [num_layouts, 4]: the sum over the layout's M replica
        rows, added left to right over m whatever the layout's index or the batch size, so the same
        layout scored anywhere gets the same bits."""
        if self.M == 1:
            return self.acc
        rows = self.acc.view(self.num_layouts, self.M, 4)
        out = rows[:, 0].clone()
        for m in range(1, self.M):
            out += rows[:, m]
        return out

    def result(self):
        """Per-layout dict of tensors with the notebook's keys (per env when M = 1)."""
        s1, s2, neg, n = self.pooled().unbind(dim=1)
        mean = s1 / n
        var = s2 / n - mean * mean  # np.var (population variance)
        low = neg / n
        w1, w2, w3 = self.weights
        return {"Average QoE": mean, "QoE Variance": var, "Low QoE Proportion": low,
                "Score": w1 * mean - w2 * var - w3 * low}

    def best(self, k: int = 1):
        """Indices (and scores) of the k best layouts, like the notebook's sort (cell 9)."""
        score = self.result()["Score"]
        top = torch.topk(score, k)
        return top.indices, top.values

    def map_result(self, stride: int = 1, load: int = 1, ue_class: int = 0):
        """Map statistics of every layout (``MComCore.layout_map`` of env row l*M for layout l: all M replica
        rows hold the same layout): dict of FP64 tensors [num_layouts] with ``result()``'s keys, over the
        grid points instead of the trajectories, plus ``Coverage`` and ``Overlap``; same threshold and
        weights."""
        env = self.env
        rows = torch.arange(0, env.num_envs, self.M, dtype=torch.int32, device=env.device)
        m = env.layout_map(rows, stride=stride, load=load, ue_class=ue_class, threshold=self.threshold, maps=False)
        return m.result(self.weights)

    def score_layouts(self, bs_xy, nbs):
        """Scores ``num_layouts`` given layouts, bs_xy int [L, B, 2] / nbs int [L], with one episode:
        resets the env and the statistics, writes layout l into its M replica rows, runs the episode
        and returns the pooled ``Score`` f32 [L].  Scoring winners on an env built with another
        ``seed`` (the UE trajectories are keyed by the movement seed) is a held-out evaluation."""
        env, L, M = self.env, self.num_layouts, self.M
        p = env.plan
        if p.bs_layout != _lib.BS_PER_ENV or p.bs_random[1] <= 0:
            raise ValueError("score_layouts needs per-env random BS layouts (config['bs_random'])")
        xy, n = check_layouts(p, bs_xy, nbs, L)
        env.reset()
        env.bs_xy.view(L, M, p.num_bs, 2).copy_(torch.from_numpy(xy).to(env.device)[:, None])
        env.nbs.view(L, M).copy_(torch.from_numpy(n).to(env.device)[:, None])
        self.reset()
        self.run_episode()
        return self.result()["Score"]


class LayoutEvolution:
    """Genetic search over per-env BS layouts: the population is the env batch (one layout per env, or
    one per M env rows with ``num_trajectories`` = M > 1), fitness is ``LayoutScorer``'s (pooled)
    ``Score`` of one whole episode, and the next population is bred on the GPU by
    ``mbe_evolve_layouts`` (DESIGN.md section 10): child c < ``elites`` is the c-th best layout copied
    verbatim, every other child comes from tournament selection (``tournament`` candidates), uniform
    slot crossover (``p_cross``), per-slot moves of at most ``step`` map units per axis (``p_move`` per
    slot), then at most one added (``p_add``) or deleted (``p_del``) BS within the scenario's
    ``bs_random`` range.  Operator randomness is Philox keyed by ``seed`` and counted by generation and
    global layout id (env_offset / M + layout), so a search is reproducible and ranks sharded with
    ``env_offset`` breed disjoint islands.

    The env must run in FORK mode with per-env layouts and ONE shared UE trajectory
    (``plan.shared_trajectory`` with movement ``reset_rng_episode``, MComCustom's default).  Only then is
    the fitness a function of the layout alone: an elite re-scored at another env index next generation
    gets bit for bit the score it had, which is what makes keeping elites sound.  With M > 1 trajectories
    every layout is scored over the same M trajectories, so the same holds for the pooled score.

    ``bs_xy`` int [L, B, 2] / ``nbs`` int [L] set the initial population of L = num_envs / M layouts
    (slots at or beyond nbs are ignored and stored as (0, 0)); by default it is the env's own random
    draw of ``reset()`` (the draw of row l*M for layout l), so generation 0 is today's random search
    over L layouts.  Defaults: tournament 4, p_cross 0.5, p_move 0.2, step 10 (5 % of MComCustom's
    200 x 200 map), p_add = p_del = 0.1, elites 1/64 of the population; of the tournament sizes 2, 3 and 4 measured in profiles/layout_evolution_bench.json, 4
    reached the best score."""

    def __init__(self, env, *, elites: int = None, tournament: int = 4, p_cross: float = 0.5,
                 p_move: float = 0.2, step: int = 10, p_add: float = 0.1, p_del: float = 0.1, seed: int = None,
                 low_qoe_threshold: float = 0.0, weights=(1.0, 0.1, 10.0), bs_xy=None, nbs=None):
        p = env.plan
        if p.mode != _lib.MODE_FORK:
            raise ValueError("LayoutEvolution needs a FORK-mode env (fitness is an episode score)")
        if p.bs_layout != _lib.BS_PER_ENV or p.bs_random[1] <= 0:
            raise ValueError("LayoutEvolution needs per-env random BS layouts (config['bs_random'])")
        if not (p.shared_trajectory and p.reset_rng_episode):
            raise ValueError("LayoutEvolution needs one UE trajectory shared by all envs and episodes "
                             "(shared_trajectory and movement reset_rng_episode): otherwise fitness depends "
                             "on the env index, not on the layout alone")
        M, B = p.num_trajectories, p.num_bs
        E = p.num_envs // M  # layouts in the population
        elites = max(1, E // 64) if elites is None else int(elites)
        if not 0 <= elites <= E:
            raise ValueError(f"elites={elites} outside 0..{E}")
        self.env, self.elites, self.M = env, elites, M
        self.scorer = LayoutScorer(env, low_qoe_threshold, weights)
        self.params = _lib.EvolveParams(seed=(p.seed if seed is None else int(seed)) & 0xFFFFFFFFFFFFFFFF,
                                        generation=0, tournament=int(tournament), step=int(step),
                                        p_cross=float(p_cross), p_move=float(p_move), p_add=float(p_add),
                                        p_del=float(p_del))
        self._xy = torch.zeros(2, E, B, 2, dtype=torch.int16, device=env.device)
        self._nbs = torch.zeros(2, E, dtype=torch.int32, device=env.device)
        self._cur = 0
        if bs_xy is None and nbs is None:
            env.reset()
            self._xy[0].copy_(env.bs_xy.view(E, M, B, 2)[:, 0])
            self._nbs[0].copy_(env.nbs.view(E, M)[:, 0])
        elif bs_xy is None or nbs is None:
            raise ValueError("an initial population needs both bs_xy and nbs")
        else:
            xy, n = check_layouts(p, bs_xy, nbs, E)
            self._xy[0].copy_(torch.from_numpy(xy))
            self._nbs[0].copy_(torch.from_numpy(n))
        self.generation = 0
        self.fitness = None  # of the last scored population (self.population())

    def population(self):
        """(bs_xy [L, B, 2], nbs [L]) that the last ``step()`` scored (the initial one before any step)."""
        i = self._cur if self.fitness is None else 1 - self._cur
        return self._xy[i], self._nbs[i]

    def step(self):
        """Scores the current population with one episode and breeds the next; returns the fitness
        tensor f32 [L] of the population just scored."""
        env, cur, M = self.env, self._cur, self.M
        L, B = self._nbs.shape[1], env.plan.num_bs
        env.reset()
        # per-env layouts are read from the bound buffers: no re-bind; layout l goes to its M replica rows
        env.bs_xy.view(L, M, B, 2).copy_(self._xy[cur][:, None])
        env.nbs.view(L, M).copy_(self._nbs[cur][:, None])
        self.scorer.reset()
        self.scorer.run_episode()
        fit = self.scorer.result()["Score"]
        elite_ids = torch.topk(torch.nan_to_num(fit, nan=-math.inf), self.elites).indices.int()
        self.params.generation = self.generation
        nxt = 1 - cur
        ptr = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
        _lib.check(env._lib.mbe_evolve_layouts(
            env._handle, ptr(fit), ptr(self._xy[cur]), ptr(self._nbs[cur]), ptr(elite_ids), self.elites,
            C.byref(self.params), ptr(self._xy[nxt]), ptr(self._nbs[nxt]), env._stream()))
        self._cur, self.fitness, self.elite_ids = nxt, fit, elite_ids
        self.generation += 1
        return fit

    def run(self, generations: int):
        """``generations`` calls of ``step``; returns each generation's best score (one sync at the end)."""
        best = [self.step().max() for _ in range(generations)]
        return torch.stack(best).cpu().tolist() if best else []

    def best(self, k: int = 1):
        """The k best layouts of the last scored population, best first, like ``LayoutScorer.best``:
        ``(bs_xy [k, B, 2], nbs [k], scores [k])``.  With elites >= 1 the best layout ever scored is
        among them."""
        if self.fitness is None:
            raise RuntimeError("best() needs at least one step()")
        top = torch.topk(torch.nan_to_num(self.fitness, nan=-math.inf), k)
        xy, nbs = self.population()
        return xy[top.indices], nbs[top.indices], self.fitness[top.indices]
