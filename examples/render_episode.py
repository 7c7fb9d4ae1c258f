#!/usr/bin/env python
"""Renders one episode of K envs as binary PPM (P6) frames, without any imaging dependency.

    python examples/render_episode.py --scenario mobile-custom-v0 --envs 4 --out frames/
    python examples/render_episode.py --best-layouts 4 --layouts 65536 --out frames/

--scenario: K envs of a registered scenario.  FORK-mode scenarios (mobile-custom-v0) record the episode
with ONE rollout(record=("pos", "assoc", "utility")) and draw all steps x envs frames with ONE
render_frames call; GYM scenarios step with random actions and draw the K envs after each step.
--best-layouts: one LayoutScorer round of MComCustom (every env a candidate BS layout, the whole episode
scored in one launch), then the K best layouts replayed over the same episode and drawn as above."""
import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mobile_env_gan_b200 as mbe  # noqa: E402
from mobile_env_gan_b200.scenarios.custom import MComCustom  # noqa: E402
from mobile_env_gan_b200.scoring import LayoutScorer  # noqa: E402


def write_ppm(path, frame):
    """frame: uint8 [H, W, 3] on the host."""
    h, w, _ = frame.shape
    with open(path, "wb") as f:
        f.write(b"P6\n%d %d\n255\n" % (w, h))
        f.write(frame.tobytes())


def write_series(frames, out, prefix, labels):
    """frames [T, K, H, W, 3] (device) -> out/<prefix>_<label>_t<step>.ppm"""
    host = frames.cpu().numpy()
    for t in range(host.shape[0]):
        for k, label in enumerate(labels):
            write_ppm(os.path.join(out, f"{prefix}_{label}_t{t:02d}.ppm"), host[t, k])
    return host.shape[0] * host.shape[1]


def fork_episode(env, envs, size):
    """One recorded episode of the bound layouts, rendered in one launch: [T, K, H, W, 3]."""
    series = env.rollout(env.plan.ep_time, record=("pos", "assoc", "utility"))
    return env.render_frames(envs, size=size, series=series)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenario", default="mobile-custom-v0")
    ap.add_argument("--envs", type=int, default=4, help="K envs of --scenario to draw")
    ap.add_argument("--best-layouts", type=int, default=0, help="K: draw the K best layouts of one search round")
    ap.add_argument("--layouts", type=int, default=1 << 16, help="candidate layouts of the search round")
    ap.add_argument("--size", type=int, nargs=2, default=None, metavar=("H", "W"))
    ap.add_argument("--out", default="frames")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    size = tuple(args.size) if args.size else None
    if args.best_layouts:
        E = (args.layouts + 31) // 32 * 32
        search = MComCustom(config={"num_envs": E})
        scorer = LayoutScorer(search)
        search.reset()
        layouts, nbs = search.bs_xy.clone(), search.nbs.clone()  # the layouts this round runs on
        scorer.run_episode()
        idx, score = scorer.best(args.best_layouts)
        # replay: the same seed and env ids redraw the same layouts and the shared UE trajectory
        replay = MComCustom(config={"num_envs": E})
        replay.reset()
        assert torch.equal(replay.bs_xy, layouts) and torch.equal(replay.nbs, nbs)
        frames = fork_episode(replay, idx, size)
        labels = [f"rank{r}_env{int(e)}" for r, e in enumerate(idx.tolist())]
        n = write_series(frames, args.out, "best", labels)
        for r, (e, s) in enumerate(zip(idx.tolist(), score.tolist())):
            print(f"rank {r}: env {e} score {s:+.4f} with {int(nbs[e])} base stations")
    else:
        env = mbe.make(args.scenario, num_envs=args.envs)
        envs = list(range(args.envs))
        if env.plan.mode == 0:  # FORK: the whole episode recorded and drawn with one launch each
            env.reset()
            frames = fork_episode(env, envs, size)
        else:  # GYM: a step needs fresh actions, so draw after each step
            env.reset()
            B, U = env.NUM_STATIONS, env.NUM_USERS
            shots = []
            for _ in range(env.plan.ep_time):
                env.step(torch.randint(0, B + 1, (env.num_envs, U), dtype=torch.int32, device=env.device))
                shots.append(env.render_frames(envs, size=size))
            frames = torch.stack(shots)
        n = write_series(frames, args.out, args.scenario, [f"env{e}" for e in envs])
    print(f"wrote {n} PPM frames to {args.out}")


if __name__ == "__main__":
    main()
