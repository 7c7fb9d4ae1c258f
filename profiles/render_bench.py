#!/usr/bin/env python
"""Throughput of the map-panel renderer (mbe_render) against the device copy bandwidth of the same run.

    python profiles/render_bench.py --out profiles/render_bench.json

Workloads: (1) mobile-medium-central, 4,096 envs at 256 x 256 (805 MB of frames per launch, more than the
126 MB L2); (2) MComCustom, one 20-step series of 1,024 envs at 256 x 256 (4.0 GB per launch).  Each is
timed with CUDA events over at least --seconds of back-to-back launches after a warm-up.  The renderer
only writes, so its output GB/s is compared with a >= 1 GB device-to-device copy_ counted as read + write
bytes (what the memory system moves for the copy)."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mobile_env_gan_b200 as mbe  # noqa: E402
from mobile_env_gan_b200.scenarios.custom import MComCustom  # noqa: E402


def timed(fn, seconds):
    """Mean seconds per call of fn over >= `seconds` of launches (CUDA events, after two warm-up calls)."""
    fn(), fn()
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    fn()
    stop.record()
    stop.synchronize()
    reps = max(3, int(seconds / max(start.elapsed_time(stop) * 1e-3, 1e-6)) + 1)
    start.record()
    for _ in range(reps):
        fn()
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop) * 1e-3 / reps, reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=0.5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "render_bench needs a CUDA device"
    dev = torch.device("cuda", 0)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    res = {"device": torch.cuda.get_device_name(dev), "nvidia_smi": q[0] if q else "unavailable"}

    n = 1 << 30  # 1 GiB
    src, dst = torch.empty(n, dtype=torch.uint8, device=dev), torch.empty(n, dtype=torch.uint8, device=dev)
    src.fill_(1)
    t, reps = timed(lambda: dst.copy_(src), args.seconds)
    copy_gbs = 2 * n / t / 1e9
    res["copy"] = {"bytes": n, "seconds_per_copy": t, "reps": reps, "gbs_read_plus_write": copy_gbs}
    del src, dst

    size = (256, 256)
    rows = []
    env = mbe.make("mobile-medium-central-v0", num_envs=4096, device=dev)
    env.reset()
    env.step(torch.randint(0, 5, (4096, 15), dtype=torch.int32, device=dev))
    frames = 4096
    fn = lambda: env.render_frames(size=size)  # noqa: E731
    rows.append(("medium-central 4096 envs", fn, frames))
    fork = MComCustom(config={"num_envs": 1024})
    fork.reset()
    series = fork.rollout(20, record=("pos", "assoc", "utility"))
    rows.append(("MComCustom 20-step series x 1024 envs", lambda: fork.render_frames(size=size, series=series),
                 20 * 1024))
    res["workloads"] = []
    for name, fn, frames in rows:
        out = fn()
        torch.cuda.synchronize()
        nbytes = out.numel()
        del out
        t, reps = timed(fn, args.seconds)
        gbs = nbytes / t / 1e9
        res["workloads"].append({"name": name, "frame": list(size), "frames": frames, "output_bytes": nbytes,
                                 "seconds_per_launch": t, "reps": reps, "frames_per_s": frames / t,
                                 "output_gbs": gbs, "frac_of_copy": gbs / copy_gbs})
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
