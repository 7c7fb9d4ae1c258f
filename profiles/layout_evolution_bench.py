#!/usr/bin/env python
"""Cost and search quality of LayoutEvolution (mbe_evolve_layouts, DESIGN.md section 10) on MComCustom.

    python profiles/layout_evolution_bench.py --out profiles/layout_evolution_bench.json

(a) One generation split into reset / copy / rollout / score+topk / evolve by CUDA events, at E = 2^16 and
    2^20 layouts (mean over --gens generations after two warm-up generations).
(b) The evolve kernel alone over --launches back-to-back launches at E = 2^20, with GB/s from the byte
    model in `evolve_bytes`, next to a device-to-device copy_ of the same population measured in the
    same run.  The 40 MB population and 4 MB fitness fit the 126 MB L2, so both read mostly from L2.
(c) Search quality: best score against layouts evaluated, evolution vs today's random search (a fresh
    Philox layout per env and round) at an equal budget of E x generations episodes, for 3 seeds.
(d) A few operator settings at E = 2^16 for 30 generations: the basis of LayoutEvolution's defaults."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mobile_env_gan_b200 import _lib  # noqa: E402
from mobile_env_gan_b200.scenarios.custom import MComCustom  # noqa: E402
from mobile_env_gan_b200.scoring import LayoutEvolution, LayoutScorer  # noqa: E402


def evolve_bytes(E, B):
    """Least DRAM/L2 traffic of one generation of children: every child writes its B-slot row and its
    count and reads one parent row and count.  Fitness reads of the tournaments and the second parent
    of a crossover are extra and not counted, so the GB/s derived from this is a lower bound."""
    return 2 * E * (4 * B + 4)


def breakdown(E, gens):
    env = MComCustom(config={"num_envs": E})
    evo = LayoutEvolution(env, seed=1)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
    names = ["reset", "copy", "rollout", "score_topk", "evolve"]
    tot = dict.fromkeys(names, 0.0)
    sc, prm = evo.scorer, evo.params
    import ctypes as C

    ptr = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    for g in range(gens + 2):  # the same sequence as LayoutEvolution.step, with events between the phases
        cur, nxt = evo._cur, 1 - evo._cur
        ev[0].record()
        env.reset()
        ev[1].record()
        env.bs_xy.copy_(evo._xy[cur])
        env.nbs.copy_(evo._nbs[cur])
        ev[2].record()
        sc.reset()
        sc.run_episode()
        ev[3].record()
        fit = sc.result()["Score"]
        elite_ids = torch.topk(torch.nan_to_num(fit, nan=-float("inf")), evo.elites).indices.int()
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
                tot[n] += ev[i].elapsed_time(ev[i + 1]) * 1e-3
    ms = {n: 1e3 * v / gens for n, v in tot.items()}
    ms["total"] = sum(ms.values())
    return {"E": E, "B": env.plan.num_bs, "generations_timed": gens, "ms_per_generation": ms,
            "evolve_over_rollout": ms["evolve"] / ms["rollout"]}


def kernel_only(E, launches):
    env = MComCustom(config={"num_envs": E})
    evo = LayoutEvolution(env, seed=2)
    evo.step()
    B = env.plan.num_bs
    import ctypes as C

    ptr = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    fit, el, prm = evo.fitness, evo.elite_ids, evo.params
    src, dst = evo._xy[0], evo._xy[1]
    sn, dn = evo._nbs[0], evo._nbs[1]

    def launch(i):
        prm.generation = 1000 + i
        _lib.check(env._lib.mbe_evolve_layouts(env._handle, ptr(fit), ptr(src), ptr(sn), ptr(el), evo.elites,
                                               C.byref(prm), ptr(dst), ptr(dn), env._stream()))

    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(10):
        launch(i)
    a.record()
    for i in range(launches):
        launch(i)
    b.record()
    b.synchronize()
    t = a.elapsed_time(b) * 1e-3 / launches
    for _ in range(10):
        dst.copy_(src)
    a.record()
    for _ in range(launches):
        dst.copy_(src)
    b.record()
    b.synchronize()
    tc = a.elapsed_time(b) * 1e-3 / launches
    nb = evolve_bytes(E, B)
    cb = 2 * src.numel() * src.element_size()
    return {"E": E, "B": B, "launches": launches, "us_per_launch": t * 1e6, "model_bytes": nb,
            "gbs": nb / t / 1e9, "copy_bytes_read_plus_write": cb, "copy_us": tc * 1e6, "copy_gbs": cb / tc / 1e9}


def quality(E, gens, seed, **ops):
    env = MComCustom(config={"num_envs": E, "seed": seed})
    evo = LayoutEvolution(env, seed=seed, **ops)
    evo_best = torch.tensor(evo.run(gens)).cummax(0).values.tolist()
    env = MComCustom(config={"num_envs": E, "seed": seed})
    sc = LayoutScorer(env)
    rnd = []
    for _ in range(gens):
        env.reset()  # next episode: a fresh Philox layout per env
        sc.reset()
        sc.run_episode()
        rnd.append(sc.result()["Score"].max())
    rnd_best = torch.stack(rnd).cpu().cummax(0).values.tolist()
    return {"seed": seed, "layouts_per_generation": E, "evolution_best": evo_best, "random_best": rnd_best}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gens", type=int, default=20, help="timed generations of (a)")
    ap.add_argument("--launches", type=int, default=500, help="timed launches of (b)")
    ap.add_argument("--quality-gens", type=int, default=50)
    ap.add_argument("--quality-envs", type=int, default=1 << 20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "layout_evolution_bench needs a CUDA device"
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    res = {"device": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}
    res["generation_breakdown"] = [breakdown(E, args.gens) for E in (1 << 16, 1 << 20)]
    print(json.dumps(res["generation_breakdown"]), flush=True)
    res["evolve_kernel"] = kernel_only(1 << 20, args.launches)
    print(json.dumps(res["evolve_kernel"]), flush=True)
    res["quality"] = [quality(args.quality_envs, args.quality_gens, s) for s in (0, 1, 2)]
    for r in res["quality"]:
        print(f"seed {r['seed']}: evolution {r['evolution_best'][-1]:.4f} random {r['random_best'][-1]:.4f}", flush=True)
    settings = [dict(tournament=2, p_cross=0.5, p_move=0.2, step=10, p_add=0.1, p_del=0.1),
                dict(tournament=3, p_cross=0.5, p_move=0.2, step=10, p_add=0.1, p_del=0.1),
                dict(tournament=4, p_cross=0.5, p_move=0.2, step=10, p_add=0.1, p_del=0.1),
                dict(tournament=3, p_cross=0.5, p_move=0.5, step=20, p_add=0.1, p_del=0.1),
                dict(tournament=3, p_cross=0.5, p_move=0.1, step=5, p_add=0.05, p_del=0.05),
                dict(tournament=3, p_cross=0.0, p_move=0.2, step=10, p_add=0.1, p_del=0.1)]
    res["settings"] = []
    for s in settings:
        r = quality(1 << 16, 30, 0, **s)
        res["settings"].append({**s, "E": 1 << 16, "generations": 30, "evolution_best": r["evolution_best"][-1],
                                "random_best": r["random_best"][-1]})
        print(json.dumps(res["settings"][-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
