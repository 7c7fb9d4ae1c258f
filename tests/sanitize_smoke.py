"""Small driver that touches every kernel family once; meant to run under
`compute-sanitizer --tool memcheck python tests/sanitize_smoke.py` on the GPU box."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mobile_env_gan_b200 as mbe  # noqa: E402
from mobile_env_gan_b200.core.schedules import ProportionalFair  # noqa: E402
from mobile_env_gan_b200.scoring import LayoutScorer  # noqa: E402


def run(env, steps, gym):
    env.reset()
    g = torch.Generator(device="cuda").manual_seed(0)
    for k in range(steps):
        if gym:
            env.step(torch.randint(0, env.plan.num_bs + 1, env.actions.shape[:2], generator=g, device="cuda",
                                   dtype=torch.int32))
        else:
            env.step(0, k)
    torch.cuda.synchronize()


for wid in ("mobile-small-central-v0", "mobile-medium-central-v0", "mobile-medium-ma-v0", "mobile-large-central-v0",
            "mobile-large-ma-v0"):
    for E in (37, 256):
        run(mbe.make(wid, num_envs=E, autoreset=True), 25, True)
        run(mbe.make(wid, num_envs=E, autoreset=True, config={"generic_kernel": True}), 25, True)
for E in (5, 129):
    env = mbe.make("mobile-custom-v0", num_envs=E, autoreset=True)
    scorer = LayoutScorer(env)
    run(env, 25, False)
    scorer.update()
    env.reset(env_mask=torch.arange(E, device="cuda") % 2 == 0)
    gen = mbe.make("mobile-custom-v0", num_envs=E, autoreset=True, config={"generic_kernel": True})
    run(gen, 25, False)
    gen.enable_debug_snr()
    gen.step(0, 0)
    gen.channel_snr(want_elig=True)
env = mbe.make("mobile-medium-ma-v0", num_envs=64)
env.reset()
for ph in (2, 1, 4, 8):
    env.stage(ph)
env.observe()
run(mbe.make("mobile-synthetic-ma-v0", num_envs=3, autoreset=True, config={"EP_MAX_TIME": 4, "arrival_params": {"ep_time": 4}}), 6, True)
run(mbe.make("mobile-medium-central-v0", num_envs=9, autoreset=True, config={"scheduler": ProportionalFair}), 25, True)
# thread-per-env FORK kernel, fused episodes (per-env and shared layouts), env windows
from mobile_env_gan_b200.scenarios import MComLarge, MComMedium, MComSmall  # noqa: E402

env = mbe.make("mobile-custom-v0", num_envs=96, autoreset=True)
run(env, 22, False)
env.rollout(23, qoe_acc=LayoutScorer(env).acc, record=("pos", "wp", "assoc", "rate", "utility"))
env.step_window(32, 32)
env.step_window(64, 17)
for cls in (MComSmall, MComMedium, MComLarge):
    fork = cls(config={"num_envs": 64, "autoreset": True, "mode": "fork"})
    run(fork, 3, False)
    # 30 x 13 has no fused episode, and a stepped episode with autoreset cannot record positions
    fork.rollout(23, qoe_acc=LayoutScorer(fork).acc, record=("rate",) if cls is MComLarge else ("pos", "rate"))
# block-per-env kernel: split phases, observe, window, central handler
big = mbe.make("mobile-synthetic-central-v0", num_envs=64, autoreset=True, config={"EP_MAX_TIME": 3, "arrival_params": {"ep_time": 3}})
run(big, 4, True)
for ph in (2, 1, 4, 8):
    big.stage(ph)
big.observe()
big.step_window(32, 32)
# host-buffer entry point
for wid in ("mobile-medium-central-v0", "mobile-medium-ma-v0"):
    h = mbe.make(wid, num_envs=6400, autoreset=True)
    h.reset()
    acts = torch.zeros(tuple(h.actions.shape), dtype=torch.int32).pin_memory()
    obs_h = torch.empty(tuple(h.obs.shape), dtype=torch.float32).pin_memory()
    rew_h = torch.empty(tuple(h.reward.shape), dtype=torch.float32).pin_memory()
    done_h = torch.empty(6400, dtype=torch.uint8).pin_memory()
    for _ in range(3):
        h.step_host(acts, obs_h, rew_h, done_h)
print("sanitize smoke done")
