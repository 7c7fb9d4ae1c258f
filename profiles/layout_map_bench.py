#!/usr/bin/env python
"""Layout maps (mbe_layout_map, DESIGN.md section 10.2) on MComCustom: what a call costs, and whether the map
score of a layout predicts its score on held-out UE trajectories.

    python profiles/layout_map_bench.py --out profiles/layout_map_bench.json

(a) Cost: MComCore.layout_map at 2^16 and 2^20 envs, strides 1 and 4, statistics only and with the three
    maps (not at 2^20 x stride 1: those maps would be 126 GB).  CUDA events, mean over --reps warm calls.
    Reported per case: BS-point tests per second (a test per connectable live BS and grid point) and the
    thread instructions per test that the integer issue rate of the card (148 SMs x 128 lanes x max SM
    clock) would allow at that rate; map bytes written per second against a device copy of 4 GiB timed in
    the same run; one call against a generation's reset + rollout of the same envs.
(b) Prediction: LayoutEvolution with M = 1 and M = 16 trajectories over 2^16 envs for --gens generations;
    its top 100 layouts are scored on --holdout trajectories of another seed, and the Spearman rank
    correlation of that held-out score with the map Score at load 1 and at load 7 is reported."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mobile_env_gan_b200.scenarios.custom import MComCustom  # noqa: E402
from mobile_env_gan_b200.scoring import LayoutEvolution, LayoutScorer  # noqa: E402

SMS, LANES = 148, 128


def timed(fn, reps):
    fn()
    fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def copy_gbs(reps):
    src = torch.empty(1 << 32, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    ms = timed(lambda: dst.copy_(src), reps)
    del src, dst
    torch.cuda.empty_cache()
    return 2 * (1 << 32) / ms / 1e6


def cost(E, reps, clock_mhz, copy):
    env = MComCustom(config={"num_envs": E})
    env.reset()
    sc = LayoutScorer(env)

    def generation():
        env.reset()
        sc.reset()
        sc.run_episode()

    rollout_ms = timed(generation, reps)
    out = []
    live = int(env.nbs.sum())  # every MComCustom BS is connectable: one test per live slot and point
    for stride in (1, 4):
        for maps in (False, True):
            if maps and E >= 1 << 20 and stride == 1:
                continue
            m = env.layout_map(stride=stride, maps=maps)
            G = m.stats[0, 0].item()
            ms = timed(lambda: env.layout_map(stride=stride, maps=maps), reps)
            tests = live * G
            rate = tests / ms * 1e3
            issue = SMS * LANES * clock_mhz * 1e6
            r = {"envs": E, "stride": stride, "maps": maps, "points_per_env": G, "ms_per_call": ms,
                 "bs_point_tests": tests, "tests_per_s": rate, "instructions_per_test_at_issue_bound": issue / rate,
                 "call_over_generation_rollout": ms / rollout_ms, "generation_reset_rollout_ms": rollout_ms}
            if maps:
                r["map_bytes"] = 3 * E * G
                r["map_gbs"] = 3 * E * G / ms / 1e6
                r["map_gbs_over_copy"] = r["map_gbs"] / copy
            out.append(r)
            print(json.dumps(r), flush=True)
            del m
    del env, sc
    torch.cuda.empty_cache()
    return out


def spearman(a, b):
    from scipy.stats import spearmanr

    return float(spearmanr(a, b).correlation)


def prediction(gens, holdout, holdout_seed):
    top = 100
    held = LayoutScorer(MComCustom(config={"num_envs": top * holdout, "seed": holdout_seed,
                                           "num_trajectories": holdout}))
    out = []
    for M in (1, 16):
        env = MComCustom(config={"num_envs": 1 << 16, "seed": 0, "num_trajectories": M})
        evo = LayoutEvolution(env, seed=0)
        evo.run(gens)
        xy, nbs, train = evo.best(top)
        test = held.score_layouts(xy, nbs).cpu()
        r = {"M": M, "layouts": (1 << 16) // M, "generations": gens, "top": top,
             "train_best": float(train[0]), "held_out_mean": float(test.mean())}
        for load in (1, 7):
            score = held.map_result(stride=1, load=load)["Score"].cpu()
            r[f"spearman_map_load{load}_vs_held_out"] = spearman(score.numpy(), test.numpy())
            r[f"map_score_load{load}_mean"] = float(score.mean())
        r["spearman_train_vs_held_out"] = spearman(train.cpu().numpy(), test.numpy())
        out.append(r)
        print(json.dumps(r), flush=True)
        del env, evo
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--gens", type=int, default=20, help="generations of the searches of (b)")
    ap.add_argument("--holdout", type=int, default=1024, help="held-out trajectories (a power of two)")
    ap.add_argument("--holdout-seed", type=int, default=12345)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "layout_map_bench needs a CUDA device"
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    res = {"device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_w_max_sm_clock_mhz": q[0] if q else None}
    clock = float(q[0].split(",")[2]) if q else float("nan")
    print(res, flush=True)
    res["copy_gbs_read_plus_write"] = copy_gbs(args.reps)
    print("device copy", res["copy_gbs_read_plus_write"], "GB/s", flush=True)
    res["cost"] = cost(1 << 16, args.reps, clock, res["copy_gbs_read_plus_write"]) + \
        cost(1 << 20, args.reps, clock, res["copy_gbs_read_plus_write"])
    res["prediction"] = {"holdout": args.holdout, "holdout_seed": args.holdout_seed,
                         "runs": prediction(args.gens, args.holdout, args.holdout_seed)}
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
