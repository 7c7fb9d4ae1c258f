#!/usr/bin/env python
"""The fork's layout search (chooseBaseStation.ipynb: run an epoch per random BS layout, score it with
`qoeValue`, keep the best) as a batched search on one B200: every env is one candidate layout, a
whole 20-step epoch is one kernel launch (mbe_rollout) and the score statistics never leave the GPU.

    python examples/layout_search.py --layouts 1000000 --rounds 5 --top 10
    torchrun --nproc-per-node 8 examples/layout_search.py --layouts 8388608   # layouts sharded over the GPUs
    python examples/layout_search.py --layouts 1048576 --generations 50       # genetic search (LayoutEvolution)
    python examples/layout_search.py --layouts 65536 --generations 10 --trajectories 8 --holdout 1024
    python examples/layout_search.py --layouts 65536 --generations 10 --holdout 1024 --map-stride 4

Multi-GPU: every rank scores its own contiguous slice of the global layout range (Philox layouts are
keyed by the global env id, so the candidates do not depend on the number of GPUs); the only exchange
is an all-gather of each rank's top-k (score, layout) rows per round.

--generations N > 0 replaces the random rounds by N generations of LayoutEvolution: each generation scores
the population, keeps the best layouts and breeds the rest from them on the GPU (mbe_evolve_layouts).
Under torchrun every rank evolves its own island (Philox counters use global env ids; no migration) and
the ranks' winners are gathered as above.

--trajectories M (a power of two) scores every layout over M UE trajectories instead of one, in the
random rounds and in the genetic search: layout l runs in the M env rows l*M .. l*M + M-1 and its score is
the notebook's qoeValue over the QoE values of all M episodes (DESIGN.md section 10).  --holdout M' then
re-scores the final top layouts on M' trajectories of another movement seed (--holdout-seed) that the
search never saw, and prints the training score next to the held-out score.  --map-stride S adds each
top layout's map statistics over every S-th map point (DESIGN.md section 10.2): the score of a UE alone
at each point, the share of points with at least one and with at least two connectable BSs.
"""
import argparse
import os
import sys
import time

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mobile_env_gan_b200.scenarios.custom import MComCustom  # noqa: E402
from mobile_env_gan_b200.scoring import LayoutEvolution, LayoutScorer  # noqa: E402
from mobile_env_gan_b200.sharding import sharded_config  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--layouts", type=int, default=1 << 20, help="candidate layouts per round (envs)")
    ap.add_argument("--rounds", type=int, default=3, help="each round draws fresh layouts (next episode)")
    ap.add_argument("--top", type=int, default=5)
    ap.add_argument("--generations", type=int, default=0, help="> 0: genetic search instead of random rounds")
    ap.add_argument("--trajectories", type=int, default=1, help="UE trajectories per layout (a power of two)")
    ap.add_argument("--holdout", type=int, default=0, help="> 0: re-score the top layouts on this many "
                    "held-out trajectories (a power of two)")
    ap.add_argument("--holdout-seed", type=int, default=1, help="scenario seed of the held-out trajectories "
                    "(the search runs MComCustom's default seed)")
    ap.add_argument("--map-stride", type=int, default=0, help="> 0: print the top layouts' map statistics "
                    "(coverage, overlap, map score) over the grid of this stride")
    args = ap.parse_args()
    M = args.trajectories
    world, rank, local = (int(os.environ.get(k, d)) for k, d in (("WORLD_SIZE", 1), ("RANK", 0), ("LOCAL_RANK", 0)))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    # whole warps of envs on every rank, and every rank's env_offset a multiple of M
    unit = max(32, M) * world
    total = (args.layouts * M + unit - 1) // unit * unit
    # autoreset: the step that ends an epoch draws the next layout, like MComCustom.reset (custom.py:40-77)
    env = MComCustom(config={"autoreset": True, "device": f"cuda:{local}", "num_trajectories": M,
                             **sharded_config(total, rank, world)})
    L, B = env.num_envs // M, env.plan.num_bs
    if args.generations > 0:
        return evolve(env, args, world, rank, total)
    scorer = LayoutScorer(env)
    env.reset()
    best = []
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for r in range(args.rounds):
        # the layouts this epoch runs on: the draw of row l*M, copied to the layout's other replica rows
        layouts, nbs = env.bs_xy.view(L, M, B, 2)[:, 0].clone(), env.nbs.view(L, M)[:, 0].clone()
        if M > 1:
            env.bs_xy.view(L, M, B, 2).copy_(layouts[:, None])
            env.nbs.view(L, M).copy_(nbs[:, None])
        scorer.reset()
        scorer.run_episode()  # one launch: 20 steps x all envs + score statistics
        idx, score = scorer.best(min(args.top, L))
        rows = torch.cat([score[:, None], nbs[idx, None].float(), layouts[idx].reshape(len(idx), -1).float()], dim=1)
        cand = gather_rows(rows, world)
        best = sorted(best + cand, key=lambda c: -c[0])[: args.top]
        if rank == 0:
            top = max(cand, key=lambda c: c[0])
            print(f"round {r}: best score {top[0]:+.4f} with {len(top[1])} base stations")
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if rank == 0:
        n = args.rounds * total
        print(f"{n // M} layouts x {M} trajectories x {env.plan.ep_time} steps on {world} GPU(s) in {dt:.3f} s = "
              f"{n * env.plan.ep_time / dt:.3e} env-steps/s (wall clock, incl. top-k and gather)")
    report(best, args, env, rank)
    if world > 1:
        dist.destroy_process_group()


def gather_rows(rows, world):
    if world > 1:  # the only exchange: every rank's top-k rows
        out = rows.new_empty((world * rows.shape[0], rows.shape[1]))
        dist.all_gather_into_tensor(out, rows.contiguous())
        rows = out
    return [(float(row[0]), row[2:2 + 2 * int(row[1])].reshape(-1, 2).int().tolist()) for row in rows.cpu()]


def report(best, args, env, rank):
    """Prints the top layouts (rank 0), with --holdout their scores on held-out trajectories beside, and with
    --map-stride their map statistics (LayoutScorer.map_result: map score, coverage, overlap)."""
    if rank != 0:
        return
    if args.holdout <= 0 and args.map_stride <= 0:
        for s, xy in best:
            print(f"{s:+.4f}  {xy}")
        return
    K, Mh, B = len(best), max(args.holdout, 1), env.plan.num_bs
    held = MComCustom(config={"device": env.device, "seed": args.holdout_seed, "num_envs": K * Mh,
                              "num_trajectories": Mh})
    xy = torch.zeros(K, B, 2, dtype=torch.int16)
    for i, (_, pts) in enumerate(best):
        xy[i, :len(pts)] = torch.tensor(pts, dtype=torch.int16)
    nbs = torch.tensor([len(pts) for _, pts in best], dtype=torch.int32)
    scorer = LayoutScorer(held)
    score = scorer.score_layouts(xy, nbs).cpu().tolist()  # also writes layout l into rows l*Mh ..
    head, cols = [f"training score ({args.trajectories} trajectories)"], [[s for s, _ in best]]
    if args.holdout > 0:
        head.append(f"held-out score ({Mh} trajectories, seed {args.holdout_seed})")
        cols.append(score)
    if args.map_stride > 0:
        r = scorer.map_result(stride=args.map_stride)
        head += [f"map score (stride {args.map_stride})", "coverage", "overlap"]
        cols += [r["Score"].cpu().tolist(), r["Coverage"].cpu().tolist(), r["Overlap"].cpu().tolist()]
    print(" | ".join(head) + " | layout")
    for i, (_, pts) in enumerate(best):
        print("  ".join(f"{c[i]:+.4f}" for c in cols) + f"  {pts}")


def evolve(env, args, world, rank, total):
    evo = LayoutEvolution(env)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for g in range(args.generations):
        fit = evo.step()
        best = fit.max().reshape(1)
        if world > 1:
            dist.all_reduce(best, op=dist.ReduceOp.MAX)
        if rank == 0:
            print(f"generation {g}: best score {float(best):+.4f}")
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    xy, nbs, score = evo.best(min(args.top, env.num_envs // args.trajectories))
    rows = torch.cat([score[:, None], nbs[:, None].float(), xy.reshape(len(score), -1).float()], dim=1)
    best = sorted(gather_rows(rows, world), key=lambda c: -c[0])[: args.top]
    if rank == 0:
        n = args.generations * total
        print(f"{n // args.trajectories} layouts x {args.trajectories} trajectories evaluated in "
              f"{args.generations} generations on {world} GPU(s) in {dt:.3f} s (wall clock, incl. the "
              f"per-generation print)")
    report(best, args, env, rank)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
