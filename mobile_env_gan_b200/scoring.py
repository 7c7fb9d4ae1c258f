"""Layout scoring (SURVEY.md 8(f)-3): the fork searches BS layouts by running an episode per
random layout and ranking them with ``qoeValue`` (mobile_env/chooseBaseStation.ipynb cell 5):

    score = w1 * mean(qoe) - w2 * var(qoe) - w3 * P(qoe < low_qoe_threshold)

over all two-decimal per-UE QoE values of the epoch (base.py:269).  With one env per layout the
whole search is a batch: ``LayoutScorer`` accumulates the statistics on the device after every
step (``mbe_accumulate_qoe``) and ranks the envs without any file round trip."""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch

from . import _lib


class LayoutScorer:
    def __init__(self, env, low_qoe_threshold: float = 0.0, weights=(1.0, 0.1, 10.0)):
        self.env, self.threshold, self.weights = env, float(low_qoe_threshold), weights
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

    def result(self):
        """Per-env dict of tensors with the notebook's keys."""
        s1, s2, neg, n = self.acc.unbind(dim=1)
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


class LayoutEvolution:
    """Genetic search over per-env BS layouts: the population is the env batch (one layout per env),
    fitness is ``LayoutScorer``'s ``Score`` of one whole episode, and the next population is bred on
    the GPU by ``mbe_evolve_layouts`` (DESIGN.md section 10): child c < ``elites`` is the c-th best
    layout copied verbatim, every other child comes from tournament selection (``tournament``
    candidates), uniform slot crossover (``p_cross``), per-slot moves of at most ``step`` map units
    per axis (``p_move`` per slot), then at most one added (``p_add``) or deleted (``p_del``) BS within
    the scenario's ``bs_random`` range.  Operator randomness is Philox keyed by ``seed`` and counted by
    generation and global env id, so a search is reproducible and ranks sharded with ``env_offset``
    breed disjoint islands.

    The env must run in FORK mode with per-env layouts and ONE shared UE trajectory
    (``plan.shared_trajectory`` with movement ``reset_rng_episode``, MComCustom's default).  Only then is
    the fitness a function of the layout alone: an elite re-scored at another env index next generation
    gets bit for bit the score it had, which is what makes keeping elites sound.

    ``bs_xy`` int [E, B, 2] / ``nbs`` int [E] set the initial population (slots at or beyond nbs are
    ignored and stored as (0, 0)); by default it is the env's own random draw of ``reset()``, so
    generation 0 is today's random search over ``num_envs`` layouts.  Defaults: tournament 4, p_cross
    0.5, p_move 0.2, step 10 (5 % of MComCustom's 200 x 200 map), p_add = p_del = 0.1, elites 1/64 of the
    population; of the tournament sizes 2, 3 and 4 measured in profiles/layout_evolution_bench.json, 4
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
        E, B = p.num_envs, p.num_bs
        elites = max(1, E // 64) if elites is None else int(elites)
        if not 0 <= elites <= E:
            raise ValueError(f"elites={elites} outside 0..{E}")
        self.env, self.elites = env, elites
        self.scorer = LayoutScorer(env, low_qoe_threshold, weights)
        self.params = _lib.EvolveParams(seed=(p.seed if seed is None else int(seed)) & 0xFFFFFFFFFFFFFFFF,
                                        generation=0, tournament=int(tournament), step=int(step),
                                        p_cross=float(p_cross), p_move=float(p_move), p_add=float(p_add),
                                        p_del=float(p_del))
        self.nmin, self.nmax = p.bs_random[0], min(p.bs_random[1], B)
        self._xy = torch.zeros(2, E, B, 2, dtype=torch.int16, device=env.device)
        self._nbs = torch.zeros(2, E, dtype=torch.int32, device=env.device)
        self._cur = 0
        if bs_xy is None and nbs is None:
            env.reset()
            self._xy[0].copy_(env.bs_xy)
            self._nbs[0].copy_(env.nbs)
        elif bs_xy is None or nbs is None:
            raise ValueError("an initial population needs both bs_xy and nbs")
        else:
            xy, n = self._check_population(bs_xy, nbs)
            self._xy[0].copy_(torch.from_numpy(xy))
            self._nbs[0].copy_(torch.from_numpy(n))
        self.generation = 0
        self.fitness = None  # of the last scored population (self.population())

    def _check_population(self, bs_xy, nbs):
        p = self.env.plan
        E, B = p.num_envs, p.num_bs
        xy = np.asarray(torch.as_tensor(bs_xy).cpu(), dtype=np.int64)
        n = np.asarray(torch.as_tensor(nbs).cpu(), dtype=np.int64)
        if xy.shape != (E, B, 2) or n.shape != (E,):
            raise ValueError(f"initial population must be bs_xy [{E}, {B}, 2] and nbs [{E}], got "
                             f"{tuple(xy.shape)} and {tuple(n.shape)}")
        if n.min() < self.nmin or n.max() > self.nmax:
            raise ValueError(f"nbs must lie in [{self.nmin}, {self.nmax}]")
        xm, ym = math.ceil(p.width) - 1, math.ceil(p.height) - 1
        live = np.arange(B)[None, :] < n[:, None]
        x, y = xy[..., 0][live], xy[..., 1][live]
        if x.size and (x.min() < 0 or x.max() > xm or y.min() < 0 or y.max() > ym):
            raise ValueError(f"BS coordinates must lie in [0, {xm}] x [0, {ym}]")
        return np.where(live[..., None], xy, 0).astype(np.int16), n.astype(np.int32)

    def population(self):
        """(bs_xy [E, B, 2], nbs [E]) that the last ``step()`` scored (the initial one before any step)."""
        i = self._cur if self.fitness is None else 1 - self._cur
        return self._xy[i], self._nbs[i]

    def step(self):
        """Scores the current population with one episode and breeds the next; returns the fitness
        tensor f32 [E] of the population just scored."""
        env, cur = self.env, self._cur
        env.reset()
        env.bs_xy.copy_(self._xy[cur])  # per-env layouts are read from the bound buffers: no re-bind
        env.nbs.copy_(self._nbs[cur])
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
