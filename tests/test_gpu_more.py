"""More GPU coverage: random shapes on the generic kernel, partial resets, observe(), state
round trips, Monitor, multi-agent 1M-env sharding slice, NCCL stats gather (needs 2 GPUs)."""
import os

import numpy as np
import pytest

from mirror import Mirror, conn_bits
from test_gpu_parity import ATOL, RTOL, close, make_env

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


@pytest.mark.parametrize("seed", range(8))
def test_random_shapes_generic_kernel(seed):
    """Shapes without a specialisation (any U, B <= 32, several BS classes) against the oracle."""
    rng = np.random.default_rng(100 + seed)
    U, B = int(rng.integers(1, 33)), int(rng.integers(1, 33))
    E = int(rng.integers(33, 400))
    handler = "ma" if seed % 2 else "central"
    bs = rng.integers(0, 200, size=(B, 2)).tolist()
    cfg = {"num_envs": E, "mode": "gym", "handler": handler, "autoreset": bool(seed % 3 == 0),
           "EP_MAX_TIME": 6, "arrival_params": {"ep_time": 6}, "ue": {"velocity": float(rng.choice([1.5, 4, 10, 12.5]))},
           "seed": int(rng.integers(0, 10**6)), "movement_params": {"reset_rng_episode": bool(seed % 2)}}
    env = make_env(bs, U, cfg)
    mir = Mirror(env)
    obs, _ = env.reset()
    close(obs.cpu().numpy().reshape(E, U, -1), mir.reset(), "reset obs")
    for k in range(14):
        acts = rng.integers(0, B + 1, size=(E, U)).astype(np.int32)
        obs, rew, _, trunc, _ = env.step(torch.from_numpy(acts).to(env.device))
        out = mir.step_gym(acts)
        assert np.array_equal(env.conn.cpu().numpy().astype(np.int64) & 0xFFFFFFFF, conn_bits(out["conn_after"])), k
        assert np.array_equal(env.pos.cpu().numpy(), out["pos_after"]), k
        assert np.array_equal(env.rate.cpu().numpy(), out["rate"]), k
        close(rew.cpu(), out["reward"], f"reward {k}")
        close(obs.cpu().numpy().reshape(E, U, -1), out["obs"], f"obs {k}")
        if not cfg["autoreset"] and out["done"].all():
            break


def test_two_bs_classes_run_on_generic_kernel_and_match_oracle_per_class():
    """BSs with different radio parameters: class-specific cut-off distance and rate table."""
    from mobile_env_gan_b200.core.base import MComCore
    from mobile_env_gan_b200.core.entities import BaseStation, UserEquipment
    from mobile_env_gan_b200.core.util import deep_dict_merge
    from oracle import mbe_oracle as orc

    config = {"num_envs": 64, "mode": "fork", "ue": {"velocity": 8}}
    cfg = deep_dict_merge(MComCore.default_config(), config)
    stations = [BaseStation(0, (60, 60), **cfg["bs"]), BaseStation(1, (140, 140), **dict(cfg["bs"], tx=30))]
    users = [UserEquipment(i, **cfg["ue"]) for i in range(9)]
    env = MComCore(stations, users, config)
    assert len(env.plan.classes) == 2
    env.reset()
    p_hi, p_lo = orc.Params(velocity=8), orc.Params(velocity=8, tx=30)
    for k in range(10):
        env.step(0, k)
        pos = env.pos.cpu().numpy().astype(np.int64)
        snr_hi, d2 = orc.batch_snr(p_hi, pos, np.array([[60, 60], [140, 140]]))
        snr_lo, _ = orc.batch_snr(p_lo, pos, np.array([[60, 60], [140, 140]]))
        snr = np.stack([snr_hi[:, :, 0], snr_lo[:, :, 1]], axis=2)
        assoc, _ = orc.batch_assoc_fork(p_hi, snr, d2)
        assert np.array_equal(env.assoc.cpu().numpy(), assoc), k
        conn = assoc[:, :, None] == np.arange(2)[None, None, :]
        n = conn.sum(axis=1, keepdims=True)
        raw = 9e6 * np.log2(1 + snr)
        with np.errstate(divide="ignore", invalid="ignore"):
            want = np.round(np.where(conn, raw / n, 0.0), 2).sum(axis=2)
        assert np.array_equal(env.rate.cpu().numpy(), want), k


def test_partial_reset_and_observe():
    bs, U = [(50, 50), (150, 50), (50, 150), (150, 150)], 15
    E = 200
    env = make_env(bs, U, {"num_envs": E, "mode": "gym", "handler": "ma", "ue": {"velocity": 5},
                           "movement_params": {"reset_rng_episode": False}})
    mir = Mirror(env)
    env.reset(), mir.reset()
    rng = np.random.default_rng(2)
    for k in range(5):
        acts = rng.integers(0, 5, size=(E, U)).astype(np.int32)
        obs, *_ = env.step(torch.from_numpy(acts).cuda())
        out = mir.step_gym(acts)
    mask = rng.random(E) < 0.3
    before = {n: getattr(env, n).clone() for n in ("pos", "wp", "conn", "t", "episode", "obs", "utility_scaled")}
    obs, _ = env.reset(env_mask=torch.from_numpy(mask).cuda())
    fresh = mir.reset(mask)
    sel = torch.from_numpy(mask).cuda()
    for n, old in before.items():  # unselected envs are untouched, bit for bit
        assert torch.equal(getattr(env, n)[~sel], old[~sel]), n
    assert np.array_equal(env.pos.cpu().numpy(), mir.pos)
    assert np.array_equal(env.t.cpu().numpy(), mir.t) and np.array_equal(env.episode.cpu().numpy(), mir.episode)
    close(obs.cpu().numpy()[mask], fresh[mask], "obs of the re-initialised envs")
    # keep stepping: both populations continue correctly
    for k in range(4):
        acts = rng.integers(0, 5, size=(E, U)).astype(np.int32)
        obs, rew, *_ = env.step(torch.from_numpy(acts).cuda())
        out = mir.step_gym(acts)
        assert np.array_equal(env.pos.cpu().numpy(), out["pos_after"])
        close(obs.cpu().numpy(), out["obs"], f"obs {k}")
    # observe() recomputes the observation of an edited state
    env.set_positions(np.broadcast_to(np.array([50, 50]), (E, U, 2)).copy())
    o = env.observe().cpu().numpy()
    assert np.allclose(o[:, :, 4], 1.0)  # standing on BS 0: its snr ratio is the maximum


def test_state_dict_replay_is_bit_identical():
    import mobile_env_gan_b200 as mbe

    env = mbe.make("mobile-medium-ma-v0", num_envs=1024, autoreset=True)
    assert len(env.action_space.spaces) == 15 and env.observation_space.spaces[0].shape == (17,)
    central = mbe.make("mobile-large-central-v0", num_envs=8)
    assert central.action_space.shape == (30,) and central.observation_space.shape == (30 * 27,)
    assert central.reset()[0].shape == (8, 30 * 27)
    env.reset()
    g = torch.Generator(device="cuda").manual_seed(0)
    acts = [torch.randint(0, 5, (1024, 15), generator=g, device="cuda", dtype=torch.int32) for _ in range(30)]
    for a in acts[:10]:
        env.step(a)
    snap = env.state_dict()
    first = []
    for a in acts[10:]:
        obs, rew, *_ = env.step(a)
        first.append((obs.clone(), rew.clone()))
    env.load_state_dict(snap)
    for a, (o, r) in zip(acts[10:], first):
        obs, rew, *_ = env.step(a)
        assert torch.equal(obs, o) and torch.equal(rew, r)


@pytest.mark.parametrize("workload,names", [
    ("mobile-medium-central-v0", {"obs", "reward", "terminated", "truncated", "metrics"}),
    ("mobile-custom-v0", {"pos", "assoc", "rate", "utility_scaled", "metrics", "done"})])
def test_bench_dumps_the_same_outputs_whatever_the_preheat(tmp_path, workload, names):
    """bench.py --dump-outputs writes what the timed path computed in its last step: the same arrays
    whatever the length of the wall-clock preheat, equal to an independent replay of the batch that step
    ran on (batch (K-1) % R from its post-reset state, with its share of the warm-up and timed steps)."""
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dumps = []
    for preheat in ("0", "0.5"):
        out = tmp_path / f"preheat{preheat}"
        cmd = [sys.executable, os.path.join(root, "bench.py"), "--workload", workload, "--envs", "32768",
               "--steps", "7", "--warmup", "3", "--no-cpu-baseline", "--preheat-seconds", preheat,
               "--dump-outputs", str(out)]
        res = subprocess.run(cmd, cwd=tmp_path, capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stderr[-2000:]
        line = json.loads(res.stdout.strip().splitlines()[-1])
        assert line["steps"] == 7 and line["repeats"] == 1
        dumps.append({p.stem: np.load(p) for p in out.glob("*.npy")})
    assert set(dumps[0]) == names
    for name, a in dumps[0].items():
        assert a.shape[0] == 32768, name
        assert a.dtype == (np.float64 if name == "rate" else np.float32), name
        assert np.array_equal(a, dumps[1][name]), name

    import bench
    import mobile_env_gan_b200 as mbe

    E, K, W = 32768, 7, 3
    fork, _, B, U = bench.workload_shape(workload)
    R = bench.rotation(workload, E)[1]
    r = (K - 1) % R
    env = mbe.make(workload, num_envs=E, device="cuda:0", autoreset=True, env_offset=r * E)
    env.reset()
    g = torch.Generator(device="cuda:0").manual_seed(1234)  # bench.py draws the actions of batches 0..R-1 in order
    for i in range(r + 1):
        acts = torch.randint(0, B + 1, (E, U), generator=g, device="cuda:0", dtype=torch.int32)
    blocks = max(2, -(-max(W, 3) // K)) + 1  # warm-up blocks + the timed block
    for i in range(blocks * sum(j % R == r for j in range(K))):
        if fork:
            env.step(0, i)
        else:
            env.step(acts)
    bench.dump_outputs(bench.step_outputs(env, fork), str(tmp_path / "replay"))
    for name, a in dumps[0].items():
        assert np.array_equal(a, np.load(tmp_path / "replay" / f"{name}.npy")), name


def test_monitor_collects_device_metrics():
    import mobile_env_gan_b200 as mbe

    env = mbe.make("mobile-custom-v0", num_envs=32)
    env.reset()
    for k in range(5):
        env.step(0, k)
        env.monitor.update(env)
    info = env.monitor.info(env=3)
    assert set(info) >= {"number connections", "number connected", "mean utility", "mean datarate"}
    scalar, _, _ = env.monitor.load_results(env=3)
    assert len(scalar) == 5 and list(scalar.columns)[:2] == ["number connections", "number connected"]
    assert scalar["number connected"].iloc[-1] == float(env.metrics[3, 1])
    v = env.view(3)
    assert len(v.userDict) == 7 and v.time == 5.0
    assert sum(len(s) for s in v.bs2ue_connections.values()) == int(env.metrics[3, 0])


def test_ma_million_env_slice_is_offset_invariant():
    """BASELINE configs[2]: 1M envs sharded 131,072 per GPU.  A slice computed as rank 5 of 8 equals
    the same global envs computed inside a differently placed shard."""
    import mobile_env_gan_b200 as mbe
    from mobile_env_gan_b200.sharding import shard_envs

    off, cnt = shard_envs(1 << 20, 5, 8)
    assert (off, cnt) == (5 * 131072, 131072)
    n = 4096
    a = mbe.make("mobile-medium-ma-v0", num_envs=n, env_offset=off + 1000, autoreset=True)
    b = mbe.make("mobile-medium-ma-v0", num_envs=n + 1000, env_offset=off, autoreset=True)
    a.reset(), b.reset()
    g = torch.Generator(device="cuda").manual_seed(4)
    for k in range(22):
        acts = torch.randint(0, 5, (n + 1000, 15), generator=g, device="cuda", dtype=torch.int32)
        oa, ra, *_ = a.step(acts[1000:])
        ob, rb, *_ = b.step(acts)
        assert torch.equal(oa, ob[1000:]) and torch.equal(ra, rb[1000:])


@pytest.mark.parametrize("wid,E", [("mobile-medium-central-v0", 96), ("mobile-medium-ma-v0", 96),
                                   ("mobile-large-central-v0", 64), ("mobile-small-ma-v0", 96),
                                   ("mobile-custom-v0", 96), ("mobile-custom-v0", 70)])
def test_soak_many_episodes_against_oracle(wid, E):
    """400 steps (20 episodes with same-step autoreset) of every default kernel family against the
    oracle: rare paths (waypoint redraws, FP64 tie fallback, re-initialisation, layout regeneration)
    are all exercised many times."""
    import mobile_env_gan_b200 as mbe

    env = mbe.make(wid, num_envs=E, autoreset=True, env_offset=777,
                   config={"movement_params": {"reset_rng_episode": False}})
    mir = Mirror(env)
    env.reset(), mir.reset()
    gym = env.actions is not None
    rng = np.random.default_rng(9)
    B, U = env.plan.num_bs, env.plan.num_ues
    for k in range(400):
        if gym:
            acts = rng.integers(0, B + 1, size=(E, U)).astype(np.int32)
            obs, rew, _, trunc, _ = env.step(torch.from_numpy(acts).cuda())
            out = mir.step_gym(acts)
            if k % 7 == 0 or out["done"].any():
                assert np.array_equal(env.conn.cpu().numpy().astype(np.int64) & 0xFFFFFFFF, conn_bits(out["conn_after"])), k
                assert np.array_equal(env.rate.cpu().numpy(), out["rate"]), k
                close(obs.cpu().numpy().reshape(E, U, -1), out["obs"], f"obs {k}")
                close(rew.cpu(), out["reward"], f"reward {k}")
        else:
            env.step(0, k)
            out = mir.step_fork()
            if k % 7 == 0 or out["done"].any():
                assert np.array_equal(env.assoc.cpu().numpy(), out["assoc"]), k
                assert np.array_equal(env.rate.cpu().numpy(), out["rate"]), k
                assert np.array_equal(env.bs_xy.cpu().numpy(), mir.bs), k
        assert np.array_equal(env.pos.cpu().numpy(), out["pos_after"]), k
    assert int(env.episode.max()) == 20


def _nccl_worker(rank, world, port, q):
    import torch.distributed as dist

    import mobile_env_gan_b200 as mbe
    from mobile_env_gan_b200.sharding import gather_episode_stats, sharded_config

    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world,
                            device_id=torch.device("cuda", rank))
    total = 1000
    cfg = sharded_config(total)
    env = mbe.make("mobile-custom-v0", device=f"cuda:{rank}", **cfg)
    env.reset()
    for k in range(3):
        env.step(0, k)
    full = gather_episode_stats(env.metrics, total)
    q.put((rank, cfg["env_offset"], full.cpu().numpy()))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_nccl_stats_gather_matches_single_gpu():
    import torch.multiprocessing as mp

    import mobile_env_gan_b200 as mbe

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29700 + os.getpid() % 200
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = [q.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    ref = mbe.make("mobile-custom-v0", num_envs=1000)
    ref.reset()
    for k in range(3):
        ref.step(0, k)
    want = ref.metrics.cpu().numpy()
    for _, _, full in got:
        assert np.array_equal(full, want)  # sharding does not change any env's result


def test_two_group_stepper_equals_whole_batch():
    """mobile_env_gan_b200.pipeline.TwoGroupStepper (two halves of one handle on two streams, each a
    dependent chain policy -> step) reproduces whole-batch stepping with the same deterministic policy."""
    import mobile_env_gan_b200 as mbe
    from mobile_env_gan_b200.pipeline import TwoGroupStepper

    E = 4096 + 64
    a = mbe.make("mobile-medium-central-v0", num_envs=E, autoreset=True)
    b = mbe.make("mobile-medium-central-v0", num_envs=E, autoreset=True)
    U, B = a.NUM_USERS, a.NUM_STATIONS

    def policy(obs, group=None):  # any deterministic function of the observation
        snr = obs.reshape(obs.shape[0], U, 2 * B + 1)[:, :, B:2 * B]
        return (snr.argmax(dim=2) + 1 + (snr.sum(dim=2) * 7).to(torch.int32) % 2).clamp_(0, B).to(torch.int32)

    a.reset(), b.reset()
    stepper = TwoGroupStepper(a)
    assert stepper.groups[0][1] % 32 == 0 and sum(n for _, n in stepper.groups) == E
    steps = 27
    stepper.run(policy, steps)
    for _ in range(steps):
        b.step(policy(b._obs_view()))
    torch.cuda.synchronize()
    for name in ("pos", "wp", "t", "episode", "conn", "rate", "utility_scaled", "obs", "reward", "done", "metrics"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name
    fork = __import__("mobile_env_gan_b200.scenarios.custom", fromlist=["MComCustom"]).MComCustom(config={"num_envs": 64})
    with pytest.raises(ValueError):
        TwoGroupStepper(fork)


def test_custom_scenario_shares_the_ue_trajectory_like_the_fork():
    """In the fork every epoch replays ONE UE trajectory (movement reset_rng_episode=True,
    base.py:130-134) over a fresh BS layout; with env index = epoch number all envs of MComCustom
    therefore share positions and waypoints while their layouts differ -- across episodes too."""
    from mobile_env_gan_b200.scenarios.custom import MComCustom

    E = 96
    env = MComCustom(config={"num_envs": E, "autoreset": True, "env_offset": 7})
    assert env.plan.shared_trajectory
    mir = Mirror(env)
    env.reset(), mir.reset()
    first_episode = []
    for k in range(45):
        env.step(0, k)
        out = mir.step_fork()
        pos = env.pos.cpu().numpy()
        assert np.array_equal(pos, out["pos_after"]), k
        assert (pos == pos[:1]).all(), k  # one trajectory for every env
        assert np.array_equal(env.bs_xy.cpu().numpy(), mir.bs) and np.array_equal(env.nbs.cpu().numpy(), mir.nbs)
        if k < 20:
            first_episode.append(pos[0].copy())
        elif k < 40:
            assert np.array_equal(pos[0], first_episode[k - 20]), k  # and for every episode
    bs = env.bs_xy.cpu().numpy()
    assert len({bs[e].tobytes() for e in range(E)}) == E  # but every env has its own layout
    own = MComCustom(config={"num_envs": E, "movement_params": {"reset_rng_episode": False}})
    assert not own.plan.shared_trajectory
    own.reset()
    own.step(0, 0)
    p = own.pos.cpu().numpy()
    assert len({p[e].tobytes() for e in range(E)}) > E // 2
    forced = MComCustom(config={"num_envs": E, "shared_trajectory": False})
    forced.reset()
    assert len({forced.pos[e].cpu().numpy().tobytes() for e in range(E)}) > E // 2


def test_bs_isolines_uses_the_reference_outline():
    """MComCore.bs_isolines (reference base.py:450-460) = Channel.isoline per BS with the default UE;
    the first BS of the small scenario is one of the golden outlines the reference produced."""
    import json

    from conftest import GOLDEN_DIR

    with open(os.path.join(GOLDEN_DIR, "isoline.json")) as f:
        gold = json.load(f)
    case = next(c for c in gold["cases"] if c["pos"] == [110, 130] and c["dthresh"] == 5.0 and c["num"] == 32)
    env = make_env([(110, 130), (65, 80), (120, 30)], 5, {"num_envs": 4})
    with np.errstate(all="ignore"):
        lines = env.bs_isolines(5.0)
    assert len(lines) == 3
    xs, ys = lines[env.stationDict[0]]
    assert list(map(float, xs)) == case["xs"] and list(map(float, ys)) == case["ys"]


def test_step_kernel_name_reports_the_dispatched_family():
    import mobile_env_gan_b200 as mbe
    from mobile_env_gan_b200.core.schedules import ProportionalFair
    from mobile_env_gan_b200.scenarios import MComSmall
    from mobile_env_gan_b200.scenarios.custom import MComCustom

    assert mbe.make("mobile-medium-central-v0", num_envs=64).step_kernel_name == "step_upt_kernel"
    assert mbe.make("mobile-large-ma-v0", num_envs=64).step_kernel_name == "step_spec_kernel"
    assert mbe.make("mobile-synthetic-central-v0", num_envs=4).step_kernel_name == "step_big_kernel"
    # a shape with a warp-segment instance still runs on the block-per-env kernel under ProportionalFair
    pf = mbe.make("mobile-medium-central-v0", num_envs=64, config={"scheduler": ProportionalFair})
    assert pf.step_kernel_name == "step_big_kernel"
    assert MComCustom(config={"num_envs": 64}).step_kernel_name == "step_tpe_fork_kernel"
    assert MComCustom(config={"num_envs": 40}).step_kernel_name == "step_spec_kernel"  # E % 32 != 0
    snr = MComCustom(config={"num_envs": 64})
    snr.enable_debug_snr()  # the debug SNR output only exists in the generic kernel
    assert snr.step_kernel_name == "step_kernel"
    # a shared layout in FORK mode: only the fused episode is thread-per-env, the step is warp-segment
    assert MComSmall(config={"num_envs": 64, "mode": "fork"}).step_kernel_name == "step_spec_kernel"
    generic = mbe.make("mobile-medium-central-v0", num_envs=64, config={"generic_kernel": True})
    assert generic.step_kernel_name == "step_kernel"


def _dispatch_env(shape, mode, handler="central", classes=1, E=64, **extra):
    """An env of one scenario shape ("custom": 7 UEs on per-env random layouts of 10 slots); classes=2
    gives BS 1 a lower transmit power, i.e. a second BS class."""
    from mobile_env_gan_b200.core.base import MComCore
    from mobile_env_gan_b200.core.entities import BaseStation, UserEquipment
    from mobile_env_gan_b200.core.util import deep_dict_merge
    from test_gpu_parity import SCENARIOS

    config = dict({"num_envs": E, "mode": mode, "handler": handler}, **extra)
    if shape == "custom":
        bs, U = [], 7
        config.update({"bs_random": (5, 10), "max_bs": 10, "ue": {"velocity": 10}})
    else:
        bs, U = SCENARIOS[shape]
    cfg = deep_dict_merge(MComCore.default_config(), config)
    stations = [BaseStation(i, tuple(xy), **dict(cfg["bs"], **({"tx": 30} if classes == 2 and i == 1 else {})))
                for i, xy in enumerate(bs)]
    env = MComCore(stations, [UserEquipment(i, **cfg["ue"]) for i in range(U)], config)
    assert len(env.plan.classes) == classes
    return env


def _step_kernels_launched(fn):
    """The libmbe step kernels fn launches, as 'name<template arguments>' without casts or blanks."""
    import re

    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    found = set()
    for ev in prof.events():
        m = re.search(r"mbe::(step_\w+<[^>]*>)", ev.name)
        if m:
            name = re.sub(r"\s+|\(int\)", "", m.group(1))
            found.add(name.replace("(bool)0", "false").replace("(bool)1", "true"))
    return found


def _shape(shape, mode, **kw):
    return lambda: _dispatch_env(shape, mode, **kw)


def _debug_snr_custom():
    from mobile_env_gan_b200.scenarios.custom import MComCustom

    env = MComCustom(config={"num_envs": 64})
    env.enable_debug_snr()  # the debug SNR output only exists in the generic kernel
    return env


def _registered(env_id, E=64, **config):
    import mobile_env_gan_b200 as mbe

    return lambda: mbe.make(env_id, num_envs=E, config=config)


def _proportional_fair():
    from mobile_env_gan_b200.core.schedules import ProportionalFair

    return _registered("mobile-medium-central-v0", scheduler=ProportionalFair)()


# (env factory, kernel of one step, kernel of a 2-step rollout or None for GYM).  One case per compiled
# whole-step or fused-episode instance, then the calls that fall back to another instance or family.
_SPEC = "step_spec_kernel<{},{},{},{},{},{}>"
_DISPATCH_CASES = {
    # thread per env: MComCustom's step and episode; the scenario shapes' FORK episodes
    "custom-fork": (_shape("custom", "fork"), "step_tpe_fork_kernel<7,10,false,false>",
                    "step_tpe_fork_kernel<7,10,true,false>"),
    "small-fork": (_shape("small", "fork"), _SPEC.format(0, 0, 5, 3, "false", "false"),
                   "step_tpe_fork_kernel<5,3,true,true>"),
    "medium-fork": (_shape("medium", "fork"), _SPEC.format(0, 0, 15, 4, "false", "false"),
                    "step_tpe_fork_kernel<15,4,true,true>"),
    # UEs per thread
    "medium-gym-central": (_shape("medium", "gym"), "step_upt_kernel<0,15,4,5>", None),
    "medium-gym-ma": (_shape("medium", "gym", handler="ma"), "step_upt_kernel<1,15,4,5>", None),
    # warp segment, shared layouts, one BS class
    "small-gym-central": (_shape("small", "gym"), _SPEC.format(1, 0, 5, 3, "false", "false"), None),
    "small-gym-ma": (_shape("small", "gym", handler="ma"), _SPEC.format(1, 1, 5, 3, "false", "false"), None),
    "large-gym-central": (_shape("large", "gym"), _SPEC.format(1, 0, 30, 13, "false", "false"), None),
    "large-gym-ma": (_shape("large", "gym", handler="ma"), _SPEC.format(1, 1, 30, 13, "false", "false"), None),
    "large-fork": (_shape("large", "fork"), _SPEC.format(0, 0, 30, 13, "false", "false"),
                   _SPEC.format(0, 0, 30, 13, "false", "false")),
    # warp segment, shared layouts, several BS classes (no one-class episode applies)
    **{f"{s}-gym-{h}-2cls": (_shape(s, "gym", handler=h, classes=2), _SPEC.format(1, int(h == "ma"), U, B, "false", "true"),
                             None)
       for s, U, B in (("small", 5, 3), ("medium", 15, 4), ("large", 30, 13)) for h in ("central", "ma")},
    **{f"{s}-fork-2cls": (_shape(s, "fork", classes=2), _SPEC.format(0, 0, U, B, "false", "true"),
                          _SPEC.format(0, 0, U, B, "false", "true"))
       for s, U, B in (("small", 5, 3), ("medium", 15, 4), ("large", 30, 13))},
    # warp segment, per-env layouts; FORK with E % 32 != 0 (the thread-per-env kernels take whole warps)
    "custom-fork-40": (_shape("custom", "fork", E=40), _SPEC.format(0, 0, 7, 10, "true", "false"),
                       _SPEC.format(0, 0, 7, 10, "true", "false")),
    "custom-gym-central": (_shape("custom", "gym"), _SPEC.format(1, 0, 7, 10, "true", "false"), None),
    "custom-gym-ma": (_shape("custom", "gym", handler="ma"), _SPEC.format(1, 1, 7, 10, "true", "false"), None),
    # fallbacks: no fused episode without whole warps, block-per-env, generic
    "small-fork-40": (_shape("small", "fork", E=40), _SPEC.format(0, 0, 5, 3, "false", "false"),
                      _SPEC.format(0, 0, 5, 3, "false", "false")),
    "synthetic": (_registered("mobile-synthetic-central-v0", E=4), "step_big_kernel<1,0,2>", None),
    "medium-proportional-fair": (_proportional_fair, "step_big_kernel<1,0,2>", None),
    "custom-debug-snr": (_debug_snr_custom, "step_kernel<0,0>", "step_kernel<0,0>"),
    "medium-generic-flag": (_registered("mobile-medium-central-v0", generic_kernel=True), "step_kernel<1,0>", None),
}


@pytest.mark.parametrize("case", list(_DISPATCH_CASES))
def test_step_and_rollout_launch_the_dispatched_instance(case):
    """The kernel instance, template arguments included, that one step (and a FORK rollout) launches."""
    from mobile_env_gan_b200 import _lib

    factory, step_kernel, rollout_kernel = _DISPATCH_CASES[case]
    env = factory()
    env.reset()
    assert step_kernel.startswith(env.step_kernel_name + "<")
    if env.plan.mode == _lib.MODE_GYM:
        actions = torch.zeros((env.num_envs, env.NUM_USERS), dtype=torch.int32, device=env.device)
        assert _step_kernels_launched(lambda: env.step(actions)) == {step_kernel}
    else:
        assert _step_kernels_launched(lambda: env.step(0, 0)) == {step_kernel}
        assert _step_kernels_launched(lambda: env.rollout(2)) == {rollout_kernel}


def test_fork_step_window_ragged_tail_and_tiny_window():
    """A window that is not a whole number of 32-env warps (or holds fewer than 32 envs) must still
    step exactly its envs: the thread-per-env FORK kernel only takes whole warps, so such windows
    fall through to the warp-segment kernel (same results bit for bit)."""
    from mobile_env_gan_b200.scenarios.custom import MComCustom

    E = 4096
    a = MComCustom(config={"num_envs": E, "autoreset": True})
    b = MComCustom(config={"num_envs": E, "autoreset": True})
    a.reset(), b.reset()
    names = ("pos", "wp", "t", "episode", "assoc", "rate", "utility_scaled", "metrics", "done", "bs_xy", "nbs")
    for s in range(23):
        before = {n: getattr(a, n).clone() for n in names}
        b.step(0, s)
        a.step_window(0, 17)          # fewer envs than one warp of the thread-per-env kernel
        a.step_window(1024, 1000)     # ragged tail: 31 warps + 8 envs
        a.step_window(2048, 2048)     # whole warps: thread-per-env kernel
        torch.cuda.synchronize()
        stepped = torch.zeros(E, dtype=torch.bool, device="cuda")
        stepped[:17] = True
        stepped[1024:2024] = True
        stepped[2048:] = True
        for n in names:
            got, want, old = getattr(a, n), getattr(b, n), before[n]
            assert torch.equal(got[stepped], want[stepped]), (n, s)
            assert torch.equal(got[~stepped], old[~stepped]), (n, s)
        # bring the untouched envs level with b for the next step
        for n in names:
            getattr(a, n).copy_(getattr(b, n))


def test_load_state_dict_rebinds_a_shared_layout_and_recomputes_obs():
    import mobile_env_gan_b200 as mbe

    env = mbe.make("mobile-small-central-v0", num_envs=256)
    ref = mbe.make("mobile-small-central-v0", num_envs=256)
    env.reset(), ref.reset()
    g = torch.Generator(device="cuda").manual_seed(3)
    acts = [torch.randint(0, 4, (256, 5), generator=g, device="cuda", dtype=torch.int32) for _ in range(12)]
    for a in acts[:4]:
        env.step(a), ref.step(a)
    snap = env.state_dict()
    obs_at_snap = env.obs.clone()
    env.set_station_positions(torch.tensor([[10, 10], [190, 190], [100, 100]]))  # another layout
    for a in acts[4:8]:
        env.step(a)
    env.load_state_dict(snap)  # back to the original layout: must re-fold it into the kernel parameters
    assert torch.equal(env.obs, obs_at_snap)
    for a in acts[4:]:
        o1, r1, *_ = env.step(a)
        o2, r2, *_ = ref.step(a)
        assert torch.equal(o1, o2) and torch.equal(r1, r2)
        assert torch.equal(env.conn, ref.conn) and torch.equal(env.rate, ref.rate)


def test_env_view_wide_shape_combines_mask_words():
    import mobile_env_gan_b200 as mbe

    env = mbe.make("mobile-synthetic-central-v0", num_envs=2)
    env.reset()
    g = torch.Generator(device="cuda").manual_seed(5)
    for _ in range(3):
        env.step(torch.randint(0, 65, (2, 512), generator=g, device="cuda", dtype=torch.int32))
    v = env.view(1)
    conn = env.conn[1].cpu().numpy().astype(np.int64) & 0xFFFFFFFF  # [U, 2]
    want = int(sum(bin(int(w)).count("1") for w in conn.reshape(-1)))
    assert sum(len(ues) for ues in v.bs2ue_connections.values()) == want
    hi = [bs.bs_id for bs, ues in v.bs2ue_connections.items() if ues and bs.bs_id >= 32]
    assert (conn[:, 1] != 0).any() == bool(hi)


def test_handle_on_another_device_does_not_change_the_current_device():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import mobile_env_gan_b200 as mbe

    torch.cuda.set_device(0)
    env = mbe.make("mobile-small-central-v0", num_envs=64, device="cuda:1")
    assert torch.cuda.current_device() == 0
    env.reset()
    with torch.cuda.device(1):
        acts = torch.zeros(64, 5, dtype=torch.int32, device="cuda:1")
    env.step(acts)
    torch.cuda.synchronize(1)
    assert torch.cuda.current_device() == 0


def test_readme_pathloss_example_runs_verbatim_and_matches_the_oracle():
    """The reference README's customisation example (README.md:108-121) against this package's module
    path: a Channel subclass that overrides power_loss only, passed through config['channel'] /
    config['channel_params'].  Connection sets, positions and FP64 rates must equal the scalar oracle
    running the same loss; observations and rewards to 1e-5."""
    import mobile_env_gan_b200 as gymnasium  # `make` with the Gymnasium ids (gymnasium itself is not a dependency)
    from mobile_env_gan_b200.core.base import MComCore
    from mobile_env_gan_b200.core.channel import Channel
    from oracle import mbe_oracle as orc

    class PathLoss(Channel):
        def __init__(self, gamma, **kwargs):
            super().__init__(**kwargs)
            # path loss exponent
            self.gamma = gamma

        def power_loss(self, bs, ue):
            """Computes power loss between BS and UE."""
            dist = bs.point.distance(ue.point)
            loss = 10 * self.gamma * np.log10(4 * np.pi * dist * bs.frequency)
            return loss

    # replace default channel model in configuration
    config = MComCore.default_config()
    config['channel'] = PathLoss

    # pass init parameters to custom channel class!
    config['channel_params'].update({'gamma': 2.0})

    # create environment with custom channel model
    config.update({"num_envs": 4, "ue": dict(config["ue"], snr_tr=3.0, velocity=9.0)})  # snr > 3: about 58 map units
    env = gymnasium.make('mobile-small-central-v0', config=config)
    # ...
    assert env.mode == "gym" and env.plan.classes[0]["log2snr_lut"] is None  # affine in log-distance: SFU path
    E, U, B = 4, env.NUM_USERS, env.NUM_STATIONS
    rng = np.random.default_rng(8)
    K = 40
    wp = rng.integers(0, 200, size=(E, U, K, 2)).astype(np.int16)
    init = rng.integers(0, 200, size=(E, U, 2)).astype(np.int16)
    init[0, 0] = env.bs_xy[0].cpu().numpy()  # a UE exactly on a BS: d = 0, log10(0) = -inf, snr = +inf
    env.reset()
    env.inject_waypoints(wp)
    env.set_positions(init)
    p = orc.Params(velocity=9.0, snr_tr=3.0, channel=("pathloss", 2.0))
    bs_xy = env.bs_xy.cpu().tolist()
    refs = []
    for e in range(E):
        r = orc.ScalarEnv(p, bs_xy, U, wp_source=lambda u, k, e=e: wp[e, u, k])
        r.reset(init[e])
        refs.append(r)
    ranged = 0
    for k in range(20):
        acts = rng.integers(0, B + 1, size=(E, U)).astype(np.int32)
        obs, rew, term, trunc, info = env.step(torch.from_numpy(acts).cuda())
        for e in range(E):
            o, r, done, inf = refs[e].step_gym(acts[e], "central")
            want = [sum(1 << b for b in c) for c in ([sorted(c) for c in refs[e].conn])]
            assert (env.conn[e].cpu().numpy().astype(np.int64) & 0xFFFFFFFF).tolist() == want, (k, e)
            assert env.pos[e].cpu().tolist() == [list(q) for q in inf["pos"]], (k, e)
            assert env.rate[e].cpu().tolist() == inf["rate"], (k, e)  # FP64, bit-exact (inf included)
            close(env.utility_scaled[e].cpu(), inf["utility"], "utility")
            close(float(rew[e]), r, "reward")
            got = obs[e].reshape(U, -1).cpu().numpy()
            fin = np.isfinite(o)  # a UE standing on a BS has snr = inf there: inf/inf in the FP64 spec
            close(got[fin], o[fin], "observation")
            ranged += sum(1 for u in range(U) for b in range(B) if not refs[e].connectable(b, u))
    assert ranged > 0  # the threshold really cut links


@pytest.mark.parametrize("handler", ["central", "ma"])
def test_step_host_reproduces_the_device_observation(handler):
    """mbe_step_host ships observations as plain FP32 rows by DMA: obs_host must equal the device
    tensor bit for bit, including the all-zero rows of finished episodes (no autoreset) and fresh rows
    after a reset."""
    import mobile_env_gan_b200 as mbe

    E = 6400
    env = mbe.make(f"mobile-medium-{handler}-v0", num_envs=E, autoreset=False)
    env.reset()
    U, B = env.NUM_USERS, env.NUM_STATIONS
    obs_h = torch.empty(tuple(env.obs.shape), dtype=torch.float32).pin_memory()
    rew_h = torch.empty(tuple(env.reward.shape), dtype=torch.float32).pin_memory()
    done_h = torch.empty(E, dtype=torch.uint8).pin_memory()
    gen = torch.Generator().manual_seed(2)
    for k in range(env.EP_MAX_TIME + 1):
        if k == env.EP_MAX_TIME:  # every env is done: reset a third of them, the rest stay inactive
            mask = (torch.arange(E) % 3 == 0)
            env.reset(env_mask=mask.cuda())
        acts = torch.randint(0, B + 1, (E, U), dtype=torch.int32, generator=gen).pin_memory()
        obs_h.fill_(7.0)
        env.step_host(acts, obs_h, rew_h, done_h)
        assert torch.equal(obs_h, env.obs.cpu()), (handler, k)
        assert torch.equal(rew_h, env.reward.cpu()) and torch.equal(done_h, env.done.cpu())
    assert bool((env.obs.view(E, -1).abs().sum(dim=1) == 0).any())  # inactive envs were part of the comparison


def test_step_host_on_a_wide_shape():
    """Two mask words per UE (40 BSs), multi-agent, block-per-env kernel, env windows."""
    from test_gpu_parity import wide_env

    env, B, U = wide_env("wide_pf", "gym", "ma", 800, autoreset=True)
    env.reset()
    obs_h = torch.empty(tuple(env.obs.shape), dtype=torch.float32).pin_memory()
    rew_h = torch.empty(tuple(env.reward.shape), dtype=torch.float32).pin_memory()
    done_h = torch.empty(800, dtype=torch.uint8).pin_memory()
    gen = torch.Generator().manual_seed(3)
    for k in range(9):
        acts = torch.randint(0, B + 1, (800, U), dtype=torch.int32, generator=gen).pin_memory()
        env.step_host(acts, obs_h, rew_h, done_h)
        assert torch.equal(obs_h, env.obs.cpu()), k
        assert torch.equal(rew_h, env.reward.cpu()) and torch.equal(done_h, env.done.cpu())
