#!/usr/bin/env python
"""Fused episode (``LayoutScorer.run_episode``: mbe_rollout, one launch where a fused kernel exists) against the
same episode as 20 ``env.step`` + ``scorer.update`` calls, for the scenario shapes in FORK mode.
    python profiles/fork_rollout_bench.py [envs]"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main(E):
    import torch

    from mobile_env_gan_b200.scenarios import MComLarge, MComMedium, MComSmall
    from mobile_env_gan_b200.scoring import LayoutScorer

    for name, cls in (("small", MComSmall), ("medium", MComMedium), ("large", MComLarge)):
        env = cls(config={"num_envs": E, "autoreset": True, "mode": "fork"})
        sc = LayoutScorer(env)
        env.reset()

        def stepped():
            for s in range(20):
                env.step(0, s)
                sc.update()

        for arm, episode in (("rollout", lambda: sc.run_episode(20)), ("step", stepped)):
            episode()
            torch.cuda.synchronize()
            before = env.launch_count
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(10):
                episode()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 10
            print(f"{arm:7s} {name:6s} E={E}: {ms:8.3f} ms per 20-step episode, "
                  f"{E * 20 / (ms * 1e-3) / 1e9:7.2f} G env-steps/s, {(env.launch_count - before) // 10} launches per episode",
                  flush=True)


if __name__ == "__main__":
    main(int(sys.argv[1]) if len(sys.argv) > 1 else 65536)
