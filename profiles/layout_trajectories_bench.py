#!/usr/bin/env python
"""Layouts scored over M UE trajectories (num_trajectories, DESIGN.md section 10) on MComCustom: what a
generation costs, and whether the layouts a search picks keep their score on trajectories it never saw.

    python profiles/layout_trajectories_bench.py --out profiles/layout_trajectories_bench.json

(a) Cost: one LayoutEvolution generation split into reset / copy / rollout / score+pool+topk / evolve by
    CUDA events at L * M = 2^20 envs for M in {1, 4, 16} (mean over --gens generations after two
    warm-up generations).
(b) Generalisation at an equal budget of 2^20 envs x --quality-gens episodes per arm: random search (a
    fresh Philox layout per env and round, one trajectory: today's search), and LayoutEvolution with
    M = 1, 4 and 16 (2^20, 2^18 and 2^16 layouts).  Each arm runs with scenario and search seeds 0, 1, 2;
    its 10 best layouts are then scored with LayoutScorer.score_layouts on --holdout trajectories of
    scenario seed --holdout-seed, which no arm trained on.  Training and held-out scores side by side."""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mobile_env_gan_b200 import _lib  # noqa: E402
from mobile_env_gan_b200.scenarios.custom import MComCustom  # noqa: E402
from mobile_env_gan_b200.scoring import LayoutEvolution, LayoutScorer  # noqa: E402

ENVS = 1 << 20
TOP = 10


def breakdown(M, gens):
    env = MComCustom(config={"num_envs": ENVS, "num_trajectories": M})
    evo = LayoutEvolution(env, seed=1)
    L, B = ENVS // M, env.plan.num_bs
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
    names = ["reset", "copy", "rollout", "score_pool_topk", "evolve"]
    tot = dict.fromkeys(names, 0.0)
    sc, prm = evo.scorer, evo.params
    ptr = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    for g in range(gens + 2):  # the same sequence as LayoutEvolution.step, with events between the phases
        cur, nxt = evo._cur, 1 - evo._cur
        ev[0].record()
        env.reset()
        ev[1].record()
        env.bs_xy.view(L, M, B, 2).copy_(evo._xy[cur][:, None])
        env.nbs.view(L, M).copy_(evo._nbs[cur][:, None])
        ev[2].record()
        sc.reset()
        sc.run_episode()
        ev[3].record()
        fit = sc.result()["Score"]
        elite_ids = torch.topk(torch.nan_to_num(fit, nan=-math.inf), evo.elites).indices.int()
        ev[4].record()
        prm.generation = evo.generation
        _lib.check(env._lib.mbe_evolve_layouts(env._handle, ptr(fit), ptr(evo._xy[cur]), ptr(evo._nbs[cur]),
                                               ptr(elite_ids), evo.elites, C.byref(prm), ptr(evo._xy[nxt]),
                                               ptr(evo._nbs[nxt]), env._stream()))
        ev[5].record()
        evo._cur, evo.fitness = nxt, fit
        evo.generation += 1
        ev[5].synchronize()
        if g >= 2:
            for i, n in enumerate(names):
                tot[n] += ev[i].elapsed_time(ev[i + 1])
    ms = {n: v / gens for n, v in tot.items()}
    ms["total"] = sum(ms.values())
    return {"envs": ENVS, "M": M, "layouts": L, "B": B, "generations_timed": gens, "ms_per_generation": ms,
            "ns_per_layout": 1e6 * ms["total"] / L}


def random_arm(seed, gens):
    env = MComCustom(config={"num_envs": ENVS, "seed": seed})
    sc = LayoutScorer(env)
    best_s = torch.empty(0, device=env.device)
    best_xy = torch.empty(0, env.plan.num_bs, 2, dtype=torch.int16, device=env.device)
    best_n = torch.empty(0, dtype=torch.int32, device=env.device)
    for _ in range(gens):
        env.reset()  # next episode: a fresh Philox layout per env, the same trajectory
        sc.reset()
        sc.run_episode()
        idx, s = sc.best(TOP)
        s, xy, n = torch.cat([best_s, s]), torch.cat([best_xy, env.bs_xy[idx]]), torch.cat([best_n, env.nbs[idx]])
        top = torch.topk(s, TOP).indices
        best_s, best_xy, best_n = s[top], xy[top], n[top]
    return best_xy, best_n, best_s


def evolution_arm(seed, gens, M):
    env = MComCustom(config={"num_envs": ENVS, "seed": seed, "num_trajectories": M})
    evo = LayoutEvolution(env, seed=seed)
    evo.run(gens)
    return evo.best(TOP)  # the elites: the best layouts ever scored


def quality(gens, holdout, holdout_seed):
    held = LayoutScorer(MComCustom(config={"num_envs": TOP * holdout, "seed": holdout_seed,
                                           "num_trajectories": holdout}))
    arms = [("random", 1, random_arm)] + [(f"evolution_M{M}", M, None) for M in (1, 4, 16)]
    out = []
    for name, M, fn in arms:
        for seed in (0, 1, 2):
            xy, nbs, train = fn(seed, gens) if fn else evolution_arm(seed, gens, M)
            test = held.score_layouts(xy, nbs)
            r = {"arm": name, "M": M, "seed": seed, "layouts_per_generation": ENVS // M, "generations": gens,
                 "train": train.cpu().tolist(), "held_out": test.cpu().tolist()}
            r["train_best"], r["held_out_of_train_best"] = r["train"][0], r["held_out"][0]
            r["train_mean_top10"] = sum(r["train"]) / TOP
            r["held_out_mean_top10"] = sum(r["held_out"]) / TOP
            r["held_out_best_of_top10"] = max(r["held_out"])
            out.append(r)
            print(f"{name:14s} seed {seed}: train best {r['train_best']:.4f} -> held-out {r['held_out_of_train_best']:.4f}"
                  f" | top-10 mean train {r['train_mean_top10']:.4f} held-out {r['held_out_mean_top10']:.4f}",
                  flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gens", type=int, default=20, help="timed generations of (a)")
    ap.add_argument("--quality-gens", type=int, default=50)
    ap.add_argument("--holdout", type=int, default=4096, help="held-out trajectories (a power of two)")
    ap.add_argument("--holdout-seed", type=int, default=12345)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "layout_trajectories_bench needs a CUDA device"
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    res = {"device": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}
    print(res, flush=True)
    res["generation_breakdown"] = [breakdown(M, args.gens) for M in (1, 4, 16)]
    for r in res["generation_breakdown"]:
        print(json.dumps(r), flush=True)
    res["holdout"] = {"trajectories": args.holdout, "seed": args.holdout_seed, "top": TOP}
    res["quality"] = quality(args.quality_gens, args.holdout, args.holdout_seed)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
