"""Parity of the CUDA path (through the C ABI, via the host mirror of MComCore) against the
oracle.  Bars (BASELINE.json north_star):
  * positions, association / connection sets, done flags, counts: bit-exact;
  * rates: bit-exact in FP64 (the per-link Shannon rate is a host-folded FP64 table indexed by
    the integer d^2, then split and rounded in FP64 on the device);
  * SNR, utility, obs, reward, mean metrics: |a-b| <= RTOL*|b| + ATOL with RTOL = 1e-5 and
    ATOL = 1e-6 (FP32 vs numpy FP64; the absolute term only matters at zero crossings of the
    [-1,1]-scaled utilities)."""
import numpy as np
import pytest

from conftest import gymref_names, load_gymref, golden_names, golden_waypoints, load_golden
from mirror import Mirror, conn_bits, conn_bool_from_words

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-5, 1e-6

torch = pytest.importorskip("torch")


def _mods():
    from mobile_env_gan_b200.core.base import MComCore
    from mobile_env_gan_b200.core.entities import BaseStation, UserEquipment

    return MComCore, BaseStation, UserEquipment


def make_env(bs_xy, nue, config):
    MComCore, BaseStation, UserEquipment = _mods()
    cfg = MComCore.default_config()
    from mobile_env_gan_b200.core.util import deep_dict_merge

    cfg = deep_dict_merge(cfg, config)
    stations = [BaseStation(i, tuple(xy), **cfg["bs"]) for i, xy in enumerate(bs_xy)] if bs_xy is not None else []
    users = [UserEquipment(i, **cfg["ue"]) for i in range(nue)]
    return MComCore(stations, users, config)


def plugin_channels():
    """The channel subclasses of the plugin fixtures, written against THIS package's Channel exactly as
    oracle/ref_harness.py:custom_channels writes them against the reference's: power_loss only
    (PathLoss is the reference README's example, README.md:108-121)."""
    from mobile_env_gan_b200.core.channels import Channel

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

    class TwoSlope(Channel):
        def __init__(self, gamma1, gamma2, d_break, **kwargs):
            super().__init__(**kwargs)
            self.gamma1, self.gamma2, self.d_break = gamma1, gamma2, d_break

        def power_loss(self, bs, ue):
            dist = bs.point.distance(ue.point)
            if dist <= self.d_break:
                return 10 * self.gamma1 * np.log10(4 * np.pi * dist * bs.frequency)
            return (10 * self.gamma1 * np.log10(4 * np.pi * self.d_break * bs.frequency)
                    + 10 * self.gamma2 * np.log10(dist / self.d_break))

    return {"pathloss": (PathLoss, ("gamma",)), "two_slope": (TwoSlope, ("gamma1", "gamma2", "d_break"))}


def env_from_record(rec, extra):
    """The env of a golden record: per-BS / per-UE parameter overrides as the reference's entity
    objects carry them (entities.py:6-57) and, when recorded, a power_loss-only Channel subclass."""
    MComCore, BaseStation, UserEquipment = _mods()
    from mobile_env_gan_b200.core.util import deep_dict_merge

    config = golden_config(rec, extra)
    chan = rec["params"].get("channel")
    if chan:
        cls, names = plugin_channels()[chan[0]]
        config["channel"] = cls
        config["channel_params"] = dict(zip(names, chan[1:]))
    cfg = deep_dict_merge(MComCore.default_config(), config)
    bs_ren = {"tx": "tx", "bw": "bw", "freq": "freq", "bs_height": "height"}
    ue_ren = {"velocity": "velocity", "snr_tr": "snr_tr", "noise": "noise", "ue_height": "height"}
    stations, users = [], []
    for i, xy in enumerate(rec["bs_xy"]):
        kw = dict(cfg["bs"])
        if rec.get("bs_over"):
            kw.update({bs_ren[k]: v for k, v in rec["bs_over"][i].items()})
        stations.append(BaseStation(i, tuple(xy), **kw))
    for i in range(len(rec["init_pos"])):
        kw = dict(cfg["ue"])
        if rec.get("ue_over"):
            kw.update({ue_ren[k]: v for k, v in rec["ue_over"][i].items()})
        users.append(UserEquipment(i, **kw))
    return MComCore(stations, users, config)


def close(a, b, what=""):
    np.testing.assert_allclose(np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64),
                               rtol=RTOL, atol=ATOL, err_msg=what)


def golden_config(rec, extra=None):
    p = rec["params"]
    cfg = {
        "width": p["width"], "height": p["height"], "EP_MAX_TIME": p["ep_time"],
        "arrival_params": {"ep_time": p["ep_time"]},
        "bs": {"bw": p["bw"], "freq": p["freq"], "tx": p["tx"], "height": p["bs_height"]},
        "ue": {"velocity": p["velocity"], "snr_tr": p["snr_tr"], "noise": p["noise"], "height": p["ue_height"]},
        "utility_params": {"lower": p["util_lower"], "upper": p["util_upper"], "coeffs": tuple(p["util_coeffs"])},
    }
    cfg.update(extra or {})
    return cfg


# ------------------------------------------------------------------ reference trajectories
@pytest.mark.parametrize("fast", [False, True])
@pytest.mark.parametrize("name", golden_names())
def test_fork_replays_reference_trajectory(name, fast):
    """Injects the reference's positions and waypoints (tests/golden, generated from the
    unmodified reference) and compares every step of the episode.  fast=False binds the debug SNR
    output, which routes the step through the generic kernel; fast=True runs whatever fused kernel
    the shape dispatches to (the specialised ones for 5x3, 15x4 and 30x13)."""
    rec = load_golden(name)
    E = 5  # replicas of the same episode: also checks envs are independent of their slot
    U = len(rec["init_pos"])
    env = env_from_record(rec, {"num_envs": E, "mode": "fork"})
    if rec.get("bs_over"):
        assert env.plan.num_bs_classes > 1
    if rec.get("ue_over"):
        assert env.plan.ue_class is not None and len(env.plan.classes) == env.plan.num_bs_classes * len(env.plan.ue_classes)
    wide = U > 32 or len(rec["bs_xy"]) > 32  # block-per-env kernel: no debug SNR output
    if wide and not fast:
        pytest.skip("wide shapes have a single kernel (covered by fast=True)")
    snr_dbg = None if fast else env.enable_debug_snr()
    seq = golden_waypoints(rec)
    K = max(1, max(len(s) for s in seq))
    wp = np.zeros((E, U, K, 2), dtype=np.int16)
    for u, s in enumerate(seq):
        for k, w in enumerate(s):
            wp[:, u, k] = w
    env.reset()
    env.inject_waypoints(wp)
    env.set_positions(np.broadcast_to(np.array(rec["init_pos"]), (E, U, 2)).copy())
    for k, g in enumerate(rec["steps"]):
        env.step(0, k)
        for e in (0, E - 1):
            assert env.pos[e].cpu().tolist() == g["pos"], (name, k)
            assert env.assoc[e].cpu().tolist() == g["conn"], (name, k)
            assert env.rate[e].cpu().tolist() == g["rate"], (name, k)  # FP64, bit-exact
            close(env.utility_scaled[e].cpu(), g["utility"], f"{name} utility step {k}")
            assert bool(env.done[e]) == g["done"]
            m = env.metrics[e].cpu().tolist()
            assert m[0] == g["n_connections"] and m[1] == g["n_connected"]
            close(m[2], g["mean_utility"], "mean utility")
            close(m[3], g["mean_datarate"], "mean datarate")
            if snr_dbg is None:
                continue
            got = snr_dbg[e].cpu().numpy().astype(np.float64)
            ref = np.array(g["snr"])
            fin = ref < 3e38  # d = 0 gives 3.8e53 in FP64 -> inf in FP32 on both sides
            close(got[fin], ref[fin], f"{name} snr step {k}")
            assert np.all(np.isinf(got[~fin]))


def test_custom_scenario_epochs_replay_reference():
    """The fork's scenario as shipped (MComCustom): env e of the batch replays epoch e of the
    reference -- its own BS layout (5..10 live slots of 10), the shared UE trajectory."""
    import json
    import os

    from conftest import GOLDEN_DIR
    from mobile_env_gan_b200.scenarios import MComCustom

    with open(os.path.join(GOLDEN_DIR, "custom_epochs.json")) as f:
        epochs = json.load(f)["epochs"]
    U, B, REP = 7, 10, 8
    epochs = [ep for ep in epochs for _ in range(REP)]  # 32 envs: the thread-per-env kernel needs E % 32 == 0
    E = len(epochs)
    for generic in (False, True):
        env = MComCustom(config={"num_envs": E, "generic_kernel": generic})
        env.reset()
        bs = np.zeros((E, B, 2), dtype=np.int16)
        nbs = np.zeros(E, dtype=np.int32)
        seqs = [golden_waypoints(ep) for ep in epochs]
        K = max(len(s) for seq in seqs for s in seq)
        wp = np.zeros((E, U, K, 2), dtype=np.int16)
        for e, ep in enumerate(epochs):
            nbs[e] = len(ep["bs_xy"])
            bs[e, : nbs[e]] = ep["bs_xy"]
            for u, s in enumerate(seqs[e]):
                for k, w in enumerate(s):
                    wp[e, u, k] = w
        env.set_station_positions(bs, nbs)
        env.inject_waypoints(wp)
        env.set_positions(np.array([ep["init_pos"] for ep in epochs]))
        for k in range(len(epochs[0]["steps"])):
            env.step(0, k)
            for e, ep in enumerate(epochs):
                g = ep["steps"][k]
                assert env.pos[e].cpu().tolist() == g["pos"], (e, k)
                assert env.assoc[e].cpu().tolist() == g["conn"], (e, k)
                assert env.rate[e].cpu().tolist() == g["rate"], (e, k)
                close(env.utility_scaled[e].cpu(), g["utility"], f"epoch {e} step {k}")
                assert bool(env.done[e]) == g["done"]


def test_custom_scenario_epochs_replay_reference_in_one_launch():
    """The same reference epochs through mbe_rollout: each whole 20-step epoch of the reference is
    ONE launch; the per-step series must be the reference's positions / association / FP64 rates."""
    import json
    import os

    from conftest import GOLDEN_DIR
    from mobile_env_gan_b200.scenarios import MComCustom

    with open(os.path.join(GOLDEN_DIR, "custom_epochs.json")) as f:
        epochs = json.load(f)["epochs"]
    U, B, REP = 7, 10, 8
    epochs = [ep for ep in epochs for _ in range(REP)]
    E, T = len(epochs), len(epochs[0]["steps"])
    env = MComCustom(config={"num_envs": E})
    env.reset()
    bs = np.zeros((E, B, 2), dtype=np.int16)
    nbs = np.zeros(E, dtype=np.int32)
    seqs = [golden_waypoints(ep) for ep in epochs]
    K = max(len(s) for seq in seqs for s in seq)
    wp = np.zeros((E, U, K, 2), dtype=np.int16)
    for e, ep in enumerate(epochs):
        nbs[e] = len(ep["bs_xy"])
        bs[e, : nbs[e]] = ep["bs_xy"]
        for u, s in enumerate(seqs[e]):
            for k, w in enumerate(s):
                wp[e, u, k] = w
    env.set_station_positions(bs, nbs)
    env.inject_waypoints(wp)
    env.set_positions(np.array([ep["init_pos"] for ep in epochs]))
    before = env.launch_count
    series = env.rollout(T, record=("pos", "assoc", "rate", "utility"))
    assert env.launch_count - before == 1
    pos, assoc, rate, util = (series[n].cpu() for n in ("pos", "assoc", "rate", "utility"))
    for e, ep in enumerate(epochs):
        for k, g in enumerate(ep["steps"]):
            assert pos[k, e].tolist() == g["pos"], (e, k)
            assert assoc[k, e].tolist() == g["conn"], (e, k)
            assert rate[k, e].tolist() == g["rate"], (e, k)  # FP64, bit-exact
            close(util[k, e], g["utility"], f"epoch {e} step {k}")
    assert bool(env.done.all())


# --------------------------------------------------------------------- FORK, Philox driven
@pytest.mark.parametrize("E", [777, 800])  # 777: warp-segment kernel (ragged tail); 800: thread-per-env kernel
@pytest.mark.parametrize("autoreset", [False, True])
def test_fork_random_layouts_match_oracle(autoreset, E):
    """MComCustom-style: random BS layout per env and episode, Philox waypoints."""
    from mobile_env_gan_b200.scenarios import MComCustom

    env = MComCustom(config={"num_envs": E, "autoreset": autoreset, "env_offset": 12345,
                             "movement_params": {"reset_rng_episode": False}})
    mir = Mirror(env)
    env.reset()
    mir.reset()
    assert np.array_equal(env.pos.cpu().numpy(), mir.pos)
    assert np.array_equal(env.nbs.cpu().numpy(), mir.nbs)
    assert np.array_equal(env.bs_xy.cpu().numpy(), mir.bs)
    for k in range(45 if autoreset else 20):
        env.step(0, k)
        out = mir.step_fork()
        assert np.array_equal(env.assoc.cpu().numpy(), out["assoc"]), k
        assert np.array_equal(env.rate.cpu().numpy(), out["rate"]), k
        assert np.array_equal(env.done.cpu().numpy().astype(bool), out["done"]), k
        assert np.array_equal(env.pos.cpu().numpy(), out["pos_after"]), k
        assert np.array_equal(env.t.cpu().numpy(), mir.t)
        assert np.array_equal(env.episode.cpu().numpy(), mir.episode)
        assert np.array_equal(env.bs_xy.cpu().numpy(), mir.bs)
        close(env.utility_scaled.cpu(), out["utility"], f"utility step {k}")
        m = env.metrics.cpu().numpy()
        assert np.array_equal(m[:, 1], out["n_connected"])
        close(m[:, 2], out["mean_utility"])
        close(m[:, 3], out["mean_datarate"])


# ----------------------------------------------------------------------------- GYM mode
SCENARIOS = {
    "small": ([(110, 130), (65, 80), (120, 30)], 5),
    "medium": ([(50, 50), (150, 50), (50, 150), (150, 150)], 15),
    "large": ([(20 + 45 * (i % 4), 25 + 50 * (i // 4)) for i in range(13)], 30),
    "wide": ([(7 * i % 200, 13 * i % 200) for i in range(32)], 32),
    "one": ([(100, 100)], 1),
}


@pytest.mark.parametrize("handler", ["central", "ma"])
@pytest.mark.parametrize("scen", list(SCENARIOS))
@pytest.mark.parametrize("autoreset", [False, True])
def test_gym_matches_oracle(scen, handler, autoreset):
    bs, U = SCENARIOS[scen]
    E = 301
    cfg = {"num_envs": E, "mode": "gym", "handler": handler, "autoreset": autoreset,
           "EP_MAX_TIME": 12, "arrival_params": {"ep_time": 12}, "ue": {"velocity": 7.5}, "seed": 99,
           "movement_params": {"reset_rng_episode": False}}
    env = make_env(bs, U, cfg)
    mir = Mirror(env)
    obs, _ = env.reset()
    ref_obs = mir.reset()
    B = len(bs)
    close(obs.cpu().numpy().reshape(E, U, -1), ref_obs, "reset obs")
    rng = np.random.default_rng(5)
    for k in range(30 if autoreset else 12):
        acts = rng.integers(0, B + 1, size=(E, U)).astype(np.int32)
        obs, rew, term, trunc, info = env.step(torch.from_numpy(acts).to(env.device))
        out = mir.step_gym(acts)
        assert np.array_equal(env.conn.cpu().numpy().astype(np.int64) & 0xFFFFFFFF, conn_bits(out["conn_after"])), k
        assert np.array_equal(env.pos.cpu().numpy(), out["pos_after"]), k
        assert np.array_equal(trunc.cpu().numpy(), out["done"]), k
        assert not term.any()
        assert np.array_equal(env.rate.cpu().numpy(), out["rate"]), k
        close(env.utility_scaled.cpu(), out["utility"], f"utility {k}")
        close(rew.cpu(), out["reward"], f"reward {k}")
        close(obs.cpu().numpy().reshape(E, U, -1), out["obs"], f"obs {k}")
        m = env.metrics.cpu().numpy()
        assert np.array_equal(m[:, 0], out["n_connections"]) and np.array_equal(m[:, 1], out["n_connected"])
        close(m[:, 3], out["mean_datarate"])


@pytest.mark.parametrize("handler", ["central", "ma"])
@pytest.mark.parametrize("name", gymref_names())
def test_gym_step_replays_reference_primitive_episodes(name, handler):
    """GYM-order episodes executed by the reference's OWN update_connections / allocateDataRate2User /
    user_total_datarates / utilities / allStationUtilities / move (tests/golden/gymref_*.json,
    oracle/ref_harness.py:record_gym_pieces_episode) replayed through the CUDA GYM step with the
    recorded actions and injected waypoints: connection sets (UEs on several BSs included),
    positions, done and FP64 rates bit-exact; utilities, reward and the broadcast BS utilities 1e-5."""
    rec = load_gymref(name)
    E, U, B = 5, len(rec["init_pos"]), len(rec["bs_xy"])
    env = env_from_record(rec, {"num_envs": E, "mode": "gym", "handler": handler})
    seq = golden_waypoints(rec)
    K = max(1, max(len(s) for s in seq))
    wp = np.zeros((E, U, K, 2), dtype=np.int16)
    for u, s in enumerate(seq):
        for k, w in enumerate(s):
            wp[:, u, k] = w
    env.reset()
    env.inject_waypoints(wp)
    env.set_positions(np.broadcast_to(np.array(rec["init_pos"]), (E, U, 2)).copy())
    F = env.plan.feature_size
    seen_bcast = 0
    for k, (acts, g) in enumerate(zip(rec["actions"], rec["steps"])):
        a = torch.tensor(acts, dtype=torch.int32, device=env.device).expand(E, U).contiguous()
        obs, rew, term, trunc, info = env.step(a)
        want_conn = [sum(1 << b for b in c) for c in g["conn_after"]]
        for e in (0, E - 1):
            assert (env.conn[e].cpu().numpy().astype(np.int64) & 0xFFFFFFFF).tolist() == want_conn, (name, k)
            assert env.pos[e].cpu().tolist() == g["pos"], (name, k)
            assert env.rate[e].cpu().tolist() == g["rate"], (name, k)  # FP64, bit-exact, multi-BS sums included
            close(env.utility_scaled[e].cpu(), g["utility"], f"{name} utility step {k}")
            assert bool(trunc[e]) == g["done"]
            m = env.metrics[e].cpu().tolist()
            assert m[0] == sum(len(c) for c in g["conn"]) and m[1] == sum(1 for c in g["conn"] if c)
            if handler == "central":
                close(float(rew[e]), float(np.mean(g["utility"])), "central reward = mean utility (metrics.py:25-28)")
            elif not g["done"]:
                # columns 2B+1 .. 3B of a multi-agent row: allStationUtilities (base.py:438-447) of the BSs
                # the UE can reach from its new position, -1 elsewhere
                row = obs[e].reshape(U, F)[:, 2 * B + 1:3 * B + 1].cpu().numpy()
                for u in range(U):
                    for b in range(B):
                        if row[u, b] != -1.0:
                            close(row[u, b], g["bs_utility"][b], f"{name} bs utility step {k}")
                            seen_bcast += 1
    assert handler == "central" or seen_bcast > 0


def test_gym_random_layouts_autoreset():
    """GYM on per-env random layouts (5..10 live BSs in 10 slots) with same-step autoreset."""
    E, U = 200, 7
    cfg = {"num_envs": E, "mode": "gym", "handler": "ma", "autoreset": True, "bs_random": (5, 10),
           "max_bs": 10, "EP_MAX_TIME": 6, "arrival_params": {"ep_time": 6}, "ue": {"velocity": 10}}
    env = make_env(None, U, cfg)
    mir = Mirror(env)
    obs, _ = env.reset()
    close(obs.cpu().numpy(), mir.reset(), "reset obs")
    rng = np.random.default_rng(11)
    for k in range(20):
        acts = rng.integers(0, 11, size=(E, U)).astype(np.int32)
        obs, rew, _, trunc, _ = env.step(torch.from_numpy(acts).to(env.device))
        out = mir.step_gym(acts)
        assert np.array_equal(env.conn.cpu().numpy().astype(np.int64) & 0xFFFFFFFF, conn_bits(out["conn_after"])), k
        assert np.array_equal(env.bs_xy.cpu().numpy(), mir.bs)
        assert np.array_equal(env.rate.cpu().numpy(), out["rate"]), k
        close(rew.cpu(), out["reward"], f"reward {k}")
        close(obs.cpu().numpy(), out["obs"], f"obs {k}")


# ------------------------------------------------------------------ stages and channel
@pytest.mark.parametrize("mode", ["fork", "gym"])
def test_split_phases_equal_fused_step(mode):
    from mobile_env_gan_b200 import _lib

    bs, U = SCENARIOS["medium"]
    cfg = {"num_envs": 256, "mode": mode, "handler": "ma", "ue": {"velocity": 4}}
    a, b = make_env(bs, U, cfg), make_env(bs, U, cfg)
    a.reset(), b.reset()
    rng = np.random.default_rng(3)
    order = [1, 2, 4] if mode == "fork" else [2, 1, 4, 8]
    for k in range(20):
        if mode == "gym":
            acts = torch.from_numpy(rng.integers(0, 5, size=(256, U)).astype(np.int32)).cuda()
            a.step(acts)
            b.actions.copy_(acts)
        else:
            a.step(0, k)
        for ph in order:
            b.stage(ph)
        for name in ("pos", "wp", "t", "rate", "utility_scaled", "done", "conn", "assoc", "obs", "reward", "metrics"):
            ta, tb = getattr(a, name), getattr(b, name)
            if ta is None:
                continue
            if name in ("obs", "reward", "metrics"):  # summation order of the fused kernel, see above
                assert torch.allclose(ta, tb, rtol=1e-6, atol=2e-6), (name, k)
            else:
                assert torch.equal(ta, tb), (name, k)
    assert _lib.PHASE_ALL == 15


@pytest.mark.parametrize("scen,mode,handler", [
    ("small", "gym", "central"), ("small", "gym", "ma"), ("medium", "gym", "central"), ("medium", "gym", "ma"),
    ("large", "gym", "central"), ("large", "gym", "ma"), ("small", "fork", "central"),
    ("medium", "fork", "central"), ("large", "fork", "central"), ("custom", "fork", "central"),
    ("custom", "gym", "ma")])
@pytest.mark.parametrize("E", [1003, 1024])
def test_specialised_kernels_equal_generic(scen, mode, handler, E):
    """The shape-specialised fused kernels (warp-segment; thread-per-env when E % 32 == 0) and the
    generic kernel share their arithmetic: every output tensor must be identical, bit for bit."""
    cfg = {"num_envs": E, "mode": mode, "handler": handler, "autoreset": True, "ue": {"velocity": 1.5},
           "EP_MAX_TIME": 9, "arrival_params": {"ep_time": 9}, "movement_params": {"reset_rng_episode": False}}
    if scen == "custom":
        bs, U = None, 7
        cfg.update({"bs_random": (5, 10), "max_bs": 10})
        B = 10
    else:
        bs, U = SCENARIOS[scen]
        B = len(bs)
    a = make_env(bs, U, cfg)
    b = make_env(bs, U, dict(cfg, generic_kernel=True))
    a.reset(), b.reset()
    g = torch.Generator(device="cuda").manual_seed(7)
    for k in range(25):
        if mode == "gym":
            acts = torch.randint(0, B + 1, (E, U), generator=g, device="cuda", dtype=torch.int32)
            a.step(acts), b.step(acts)
        else:
            a.step(0, k), b.step(0, k)
        for name in ("pos", "wp", "t", "episode", "rate", "utility_scaled", "done", "conn", "assoc", "obs",
                     "reward", "metrics", "bs_xy", "nbs"):
            ta, tb = getattr(a, name), getattr(b, name)
            if ta is None:
                continue
            if name in ("obs", "reward", "metrics"):
                # per-env float sums: the several-UEs-per-thread kernels add in a different (fixed)
                # order than the shuffle tree, so the last ulp may differ
                assert torch.allclose(ta, tb, rtol=1e-6, atol=2e-6), (name, k)
            else:
                assert torch.equal(ta, tb), (name, k)


def test_movement_fast_path_is_exact():
    """The FP32 fast path of the movement falls back to the reference's FP64 chain near rounding
    ties; positions must equal the oracle for awkward velocities (exact .5 ties with v=1.5)."""
    for v in (1.5, 0.5, 2.5, 3.0, 7.5, 10, 12.25, 33.3):
        env = make_env(SCENARIOS["medium"][0], 15, {"num_envs": 4096, "mode": "fork", "ue": {"velocity": v},
                                                    "EP_MAX_TIME": 60, "arrival_params": {"ep_time": 60}})
        mir = Mirror(env)
        env.reset(), mir.reset()
        for k in range(60):
            env.step(0, k)
            out = mir.step_fork()
            assert np.array_equal(env.pos.cpu().numpy(), out["pos_after"]), (v, k)


def test_channel_kernel_matches_oracle():
    from oracle import mbe_oracle as orc

    bs, U = SCENARIOS["large"]
    env = make_env(bs, U, {"num_envs": 1000, "mode": "fork", "ue": {"velocity": 10}})
    mir = Mirror(env)
    env.reset(), mir.reset()
    for k in range(3):
        env.step(0, k), mir.step_fork()
    snr, elig = env.channel_snr(want_elig=True)
    ref, _ = orc.batch_snr(mir.p, mir.pos, mir.bs)
    got = snr.cpu().numpy().astype(np.float64)
    fin = ref < 3e38  # d = 0: 3.8e53 in FP64, inf in FP32
    assert np.all(np.isinf(got[~fin]))
    rel = np.abs(got[fin] - ref[fin]) / ref[fin]
    assert rel.max() <= RTOL, f"max rel err {rel.max():.3e}"
    assert np.array_equal(elig.cpu().numpy().astype(np.int64) & 0xFFFFFFFF, conn_bits(ref > mir.p.snr_tr))


# ------------------------------------------------------------------------- full size
def _compiled_oracle():
    """oracle/c_oracle.CEnvBatch, or skip when the C restatement cannot be built / loaded here."""
    try:
        from oracle import c_oracle

        c_oracle.load()
    except Exception as exc:  # noqa: BLE001 - no gcc and no prebuilt library on this box
        pytest.skip(f"compiled oracle unavailable: {exc}")
    return c_oracle.CEnvBatch


def _rates_bit_exact(got, want, what):
    """FP64 rates against the compiled restatement fed with the numpy snr / rate tables of the pinned oracle
    (``CEnvBatch(pinned_tables=True)``): bit equality for every env of the full-size batch.  (On its own
    glibc chain the C file differs from numpy in the last ulp of a few values, i.e. a handful of 0.01
    rounding flips per million rates -- tests/test_c_oracle.py keeps that independent chain pinned.)"""
    got, want = np.asarray(got), np.asarray(want)
    assert np.array_equal(got, want), (what, int((got != want).sum()), float(np.abs(got - want).max(initial=0.0)))


@pytest.mark.parametrize("env_id,E", [("mobile-medium-central-v0", 65536), ("mobile-medium-ma-v0", 131072)])
def test_full_size_gym_episode_matches_compiled_oracle(env_id, E):
    """BASELINE configs[1] / configs[2] at FULL size against the compiled restatement of the reference's
    arithmetic (oracle/mbe_oracle_c.c, pinned to the reference fixtures by tests/test_c_oracle.py): a
    whole Philox-driven episode of every env -- connection sets, positions and done exact, rates bit-exact, utilities / rewards / observations to 1e-5."""
    import mobile_env_gan_b200 as mbe

    CEnvBatch = _compiled_oracle()
    env = mbe.make(env_id, num_envs=E)
    mir = Mirror(env)
    env.reset()
    mir._reinit(np.ones(E, dtype=bool))
    U, B = mir.U, mir.B
    assert np.array_equal(env.pos.cpu().numpy(), mir.pos)
    c = CEnvBatch(mir.p, mir.bs, E, U, handler=mir.handler, pinned_tables=True)
    c.reset(mir.pos)
    rng = np.random.default_rng(E)
    for k in range(env.plan.ep_time):
        acts = rng.integers(0, B + 1, size=(E, U)).astype(np.int32)
        mir.t = c.t.astype(np.int64)
        c.step_gym(acts, mir.new_wp())
        obs, rew, _, trunc, _ = env.step(torch.from_numpy(acts).to(env.device))
        assert np.array_equal(conn_bool_from_words(env.conn.cpu().numpy(), B), c.conn.astype(bool)), k
        assert np.array_equal(env.pos.cpu().numpy(), c.pos), k
        assert np.array_equal(trunc.cpu().numpy(), c.done.astype(bool)), k
        _rates_bit_exact(env.rate.cpu().numpy(), c.rate, f"rate step {k}")
        close(env.utility_scaled.cpu(), c.util, f"utility {k}")
        close(rew.cpu(), c.reward, f"reward {k}")
        close(obs.cpu().numpy().reshape(E, U, -1), c.obs, f"obs {k}")
    assert bool(trunc.all())


def test_full_size_fork_custom_episode_matches_compiled_oracle():
    """The fork's own scenario at 262,144 envs (random per-env layouts, shared UE trajectory): a whole
    episode against the compiled restatement -- association, positions, done exact, rates bit-exact."""
    from mobile_env_gan_b200.scenarios.custom import MComCustom

    CEnvBatch = _compiled_oracle()
    E = 262144
    env = MComCustom(config={"num_envs": E})
    mir = Mirror(env)
    env.reset()
    mir._reinit(np.ones(E, dtype=bool))
    assert np.array_equal(env.bs_xy.cpu().numpy(), mir.bs) and np.array_equal(env.nbs.cpu().numpy(), mir.nbs)
    c = CEnvBatch(mir.p, mir.bs, E, mir.U, nbs=mir.nbs, pinned_tables=True)
    c.reset(mir.pos)
    for k in range(env.plan.ep_time):
        mir.t = c.t.astype(np.int64)
        c.step_fork(mir.new_wp())
        env.step(0, k)
        assert np.array_equal(env.assoc.cpu().numpy(), c.assoc), k
        assert np.array_equal(env.pos.cpu().numpy(), c.pos), k
        assert np.array_equal(env.done.cpu().numpy(), c.done), k
        _rates_bit_exact(env.rate.cpu().numpy(), c.rate, f"rate step {k}")
        close(env.utility_scaled.cpu(), c.util, f"utility {k}")
        m = env.metrics.cpu().numpy()
        assert np.array_equal(m[:, 1], c.metrics[:, 1]), k
    assert bool(env.done.all())


def test_full_size_medium_properties_and_sharding():
    """BASELINE configs[1] size (65,536 envs): sharded halves reproduce the whole, and the
    size-independent invariants of the domain hold."""
    import mobile_env_gan_b200 as mbe

    E = 65536
    whole = mbe.make("mobile-medium-central-v0", num_envs=E, autoreset=True)
    lo = mbe.make("mobile-medium-central-v0", num_envs=E // 2, autoreset=True)
    hi = mbe.make("mobile-medium-central-v0", num_envs=E // 2, autoreset=True, env_offset=E // 2)
    for env in (whole, lo, hi):
        env.reset()
    g = torch.Generator(device="cuda").manual_seed(1)
    U, B = 15, 4
    for k in range(25):
        acts = torch.randint(0, B + 1, (E, U), generator=g, device="cuda", dtype=torch.int32)
        _, elig_pre = whole.channel_snr(want_elig=True)
        obs, rew, _, trunc, _ = whole.step(acts)
        o1, r1, _, t1, _ = lo.step(acts[: E // 2])
        o2, r2, _, t2, _ = hi.step(acts[E // 2:])
        assert torch.equal(obs, torch.cat([o1, o2])) and torch.equal(rew, torch.cat([r1, r2]))
        assert torch.equal(trunc, torch.cat([t1, t2]))
        assert bool(trunc.all()) == ((k + 1) % 20 == 0) and bool(trunc.any()) == bool(trunc.all())
        assert float(obs.min()) >= -1.0 and float(obs.max()) <= 1.0
        assert float(rew.min()) >= -1.0 and float(rew.max()) <= 1.0
        assert int((whole.conn & ~elig_pre).count_nonzero()) == 0  # links only where connectable (base.py:221-227)
        if not bool(trunc.any()):  # on the last step the links are dropped but the rates are the step's
            con = whole.conn != 0
            assert bool((whole.rate[con] > 0).all()) and bool((whole.rate[~con] == 0).all())
        o = obs.view(E, U, 2 * B + 1)
        assert torch.equal(o[:, :, :B] > 0, ((whole.conn.unsqueeze(-1) >> torch.arange(B, device="cuda")) & 1) > 0)
        assert float(o[:, :, B:2 * B].max(dim=2).values.min()) == 1.0  # the best BS has ratio 1


def test_step_host_roundtrip():
    import mobile_env_gan_b200 as mbe

    E, U, B = 4096, 15, 4
    a = mbe.make("mobile-medium-central-v0", num_envs=E)
    b = mbe.make("mobile-medium-central-v0", num_envs=E)
    a.reset(), b.reset()
    acts = torch.randint(0, B + 1, (E, U), dtype=torch.int32).pin_memory()
    obs_h = torch.empty(E, U * (2 * B + 1), dtype=torch.float32).pin_memory()
    rew_h = torch.empty(E, dtype=torch.float32).pin_memory()
    done_h = torch.empty(E, dtype=torch.uint8).pin_memory()
    a.step_host(acts, obs_h, rew_h, done_h)
    obs, rew, _, trunc, _ = b.step(acts.cuda())
    torch.cuda.synchronize()
    assert torch.equal(obs_h, obs.cpu()) and torch.equal(rew_h, rew.cpu()) and torch.equal(done_h.bool(), trunc.cpu())


@pytest.mark.parametrize(
    "env_id,E",
    [
        ("mobile-medium-central-v0", 7000),  # UEs-per-thread kernel, ragged last window
        ("mobile-medium-ma-v0", 6144),
        ("mobile-small-central-v0", 9001),  # specialised warp-segment kernel
        ("mobile-large-ma-v0", 6500),
    ],
)
def test_step_host_windows_match_device_step(env_id, E):
    """mbe_step_host splits a batch with observations into env windows on two streams (copy/step
    overlap), and mbe_step_window steps a sub-range: both must reproduce the single whole-batch launch
    exactly, over a full episode + autoreset."""
    import mobile_env_gan_b200 as mbe

    a = mbe.make(env_id, num_envs=E, autoreset=True)  # host windows
    b = mbe.make(env_id, num_envs=E, autoreset=True)  # one launch
    c = mbe.make(env_id, num_envs=E, autoreset=True)  # explicit windows on two streams
    a.reset(), b.reset(), c.reset()
    U, B = a.NUM_USERS, a.NUM_STATIONS
    ma = "-ma-" in env_id
    obs_h = torch.empty(tuple(a.obs.shape), dtype=torch.float32).pin_memory()
    rew_h = torch.empty((E, U) if ma else (E,), dtype=torch.float32).pin_memory()
    done_h = torch.empty(E, dtype=torch.uint8).pin_memory()
    gen = torch.Generator().manual_seed(E)
    first_launches = a.launch_count
    steps = a.EP_MAX_TIME + 3
    side = torch.cuda.Stream()
    cut = (E // 3) // 32 * 32
    for _ in range(steps):
        acts = torch.randint(0, B + 1, (E, U), dtype=torch.int32, generator=gen).pin_memory()
        a.step_host(acts, obs_h, rew_h, done_h)
        b.step(acts.cuda())
        c.actions.copy_(acts.cuda())
        torch.cuda.synchronize()
        c.step_window(cut, E - cut, stream=side)
        c.step_window(0, cut)
        torch.cuda.synchronize()
        assert torch.equal(obs_h.view(-1), b.obs.cpu().view(-1))
        assert torch.equal(rew_h.view(-1), b.reward.cpu().view(-1))
        assert torch.equal(done_h, b.done.cpu())
        for name in ("pos", "wp", "t", "episode", "conn", "rate", "utility_scaled", "metrics", "obs", "reward", "done"):
            assert torch.equal(getattr(a, name), getattr(b, name)), name
            assert torch.equal(getattr(c, name), getattr(b, name)), name
    assert a.launch_count - first_launches == min(4, E // 3072) * steps  # windows hold >= 3072 envs


def test_step_host_matches_device_step_fork_custom():
    """mbe_step_host in FORK mode (one window: no observations to download) reproduces the device step
    for the fork's own scenario (thread-per-env FORK kernel, per-env random layouts)."""
    from mobile_env_gan_b200.scenarios.custom import MComCustom

    E = 8192
    a = MComCustom(config={"num_envs": E, "autoreset": True})
    b = MComCustom(config={"num_envs": E, "autoreset": True})
    a.reset(), b.reset()
    done_h = torch.empty(E, dtype=torch.uint8).pin_memory()
    first_launches = a.launch_count
    for s in range(23):
        a.step_host(None, None, None, done_h)
        b.step(0, s)
        torch.cuda.synchronize()
        assert torch.equal(done_h, b.done.cpu())
        for name in ("pos", "wp", "t", "episode", "assoc", "rate", "utility_scaled", "metrics", "bs_xy", "nbs"):
            assert torch.equal(getattr(a, name), getattr(b, name)), name
    assert a.launch_count - first_launches == 23


# ------------------------------------------------- wide shapes / ProportionalFair (block-per-env)
WIDE = {
    # name: (B, U, map, scheduler)
    "wide_rf": (40, 70, 200, "rf"),
    "wide_pf": (40, 70, 200, "pf"),
    "medium_pf": (4, 15, 200, "pf"),
    "medium_ratefair": (4, 15, 200, "ratefair"),
    "wide_ratefair": (40, 70, 200, "ratefair"),
    "synthetic": (64, 512, 800, "pf"),  # BASELINE.json configs[4]
    "many_ue": (8, 1024, 300, "rf"),
}


def wide_env(name, mode, handler, E, autoreset, extra=None):
    from mobile_env_gan_b200.core.schedules import ProportionalFair, RateFair, ResourceFair

    B, U, size, sched = WIDE[name]
    rng = np.random.default_rng(B * 1000 + U)
    bs = rng.integers(0, size, size=(B, 2)).tolist()
    cfg = {"num_envs": E, "mode": mode, "handler": handler, "autoreset": autoreset, "width": size, "height": size,
           "movement_params": {"width": size, "height": size, "reset_rng_episode": False},
           "EP_MAX_TIME": 7, "arrival_params": {"ep_time": 7}, "ue": {"velocity": 9},
           "scheduler": {"pf": ProportionalFair, "rf": ResourceFair, "ratefair": RateFair}[sched]}
    cfg.update(extra or {})
    return make_env(bs, U, cfg), B, U


@pytest.mark.parametrize("handler", ["central", "ma"])
@pytest.mark.parametrize("name", list(WIDE))
def test_wide_gym_matches_oracle(name, handler):
    E = 24 if name in ("synthetic", "many_ue") else 96
    env, B, U = wide_env(name, "gym", handler, E, autoreset=True)
    mir = Mirror(env)
    obs, _ = env.reset()
    close(obs.cpu().numpy().reshape(E, U, -1), mir.reset(), "reset obs")
    rng = np.random.default_rng(17)
    for k in range(16):
        acts = rng.integers(0, B + 1, size=(E, U)).astype(np.int32)
        obs, rew, _, trunc, _ = env.step(torch.from_numpy(acts).to(env.device))
        out = mir.step_gym(acts)
        assert np.array_equal(conn_bool_from_words(env.conn.cpu().numpy(), B), out["conn_after"]), k
        assert np.array_equal(env.pos.cpu().numpy(), out["pos_after"]), k
        assert np.array_equal(trunc.cpu().numpy(), out["done"]), k
        assert np.array_equal(env.rate.cpu().numpy(), out["rate"]), k  # FP64, bit-exact (RF and PF)
        close(env.utility_scaled.cpu(), out["utility"], f"utility {k}")
        close(rew.cpu(), out["reward"], f"reward {k}")
        close(obs.cpu().numpy().reshape(E, U, -1), out["obs"], f"obs {k}")
        m = env.metrics.cpu().numpy()
        assert np.array_equal(m[:, 0], out["n_connections"]) and np.array_equal(m[:, 1], out["n_connected"])
        close(m[:, 2], out["mean_utility"])
        close(m[:, 3], out["mean_datarate"])


def test_synthetic_shape_many_envs_matches_compiled_oracle():
    """BASELINE configs[4] shape (64 BS x 512 UE, ProportionalFair) on 1,024 envs against the compiled
    restatement (the numpy oracle above is limited to 24 envs by its speed): connection sets, positions,
    done and FP64 rates exact, utilities / reward / observations 1e-5."""
    CEnvBatch = _compiled_oracle()
    E = 1024
    env, B, U = wide_env("synthetic", "gym", "central", E, autoreset=False)
    mir = Mirror(env)
    env.reset()
    mir._reinit(np.ones(E, dtype=bool))
    c = CEnvBatch(mir.p, mir.bs, E, U, handler="central", pinned_tables=True)
    c.reset(mir.pos)
    rng = np.random.default_rng(3)
    for k in range(3):
        acts = rng.integers(0, B + 1, size=(E, U)).astype(np.int32)
        mir.t = c.t.astype(np.int64)
        c.step_gym(acts, mir.new_wp())
        obs, rew, _, trunc, _ = env.step(torch.from_numpy(acts).to(env.device))
        assert np.array_equal(conn_bool_from_words(env.conn.cpu().numpy(), B), c.conn.astype(bool)), k
        assert np.array_equal(env.pos.cpu().numpy(), c.pos), k
        assert np.array_equal(trunc.cpu().numpy(), c.done.astype(bool)), k
        _rates_bit_exact(env.rate.cpu().numpy(), c.rate, f"rate step {k}")
        close(env.utility_scaled.cpu(), c.util, f"utility {k}")
        close(rew.cpu(), c.reward, f"reward {k}")
        close(obs.cpu().numpy().reshape(E, U, -1), c.obs, f"obs {k}")


@pytest.mark.parametrize("name", ["wide_rf", "wide_pf", "many_ue"])
def test_wide_fork_matches_oracle(name):
    E = 40
    env, B, U = wide_env(name, "fork", "central", E, autoreset=False)
    mir = Mirror(env)
    env.reset(), mir.reset()
    for k in range(7):
        env.step(0, k)
        out = mir.step_fork()
        assert np.array_equal(env.assoc.cpu().numpy(), out["assoc"]), k
        assert np.array_equal(env.rate.cpu().numpy(), out["rate"]), k
        assert np.array_equal(env.pos.cpu().numpy(), out["pos_after"]), k
        assert np.array_equal(env.done.cpu().numpy().astype(bool), out["done"]), k
        close(env.utility_scaled.cpu(), out["utility"], f"utility {k}")
        m = env.metrics.cpu().numpy()
        assert np.array_equal(m[:, 1], out["n_connected"])
        close(m[:, 3], out["mean_datarate"])


def test_wide_connection_mask_has_two_words():
    env, B, U = wide_env("wide_rf", "gym", "central", 8, autoreset=False)
    assert env.plan.num_ues == 70 and env.conn.dim() == 3 and env.conn.shape[2] == 2


def test_layout_scorer_matches_notebook_formula():
    """chooseBaseStation.ipynb cell 5 `qoeValue` over the oracle's two-decimal QoE values."""
    from mobile_env_gan_b200.scenarios import MComCustom
    from mobile_env_gan_b200.scoring import LayoutScorer

    E = 500
    env = MComCustom(config={"num_envs": E})
    mir = Mirror(env)
    scorer = LayoutScorer(env)
    env.reset(), mir.reset()
    qoe = []
    for k in range(20):
        env.step(0, k)
        scorer.update()
        qoe.append(np.round(mir.step_fork()["utility"], 2))
    all_qoe = np.concatenate(qoe, axis=1)  # [E, T*U]
    want = all_qoe.mean(axis=1) - 0.1 * all_qoe.var(axis=1) - 10.0 * (all_qoe < 0.0).mean(axis=1)
    got = scorer.result()
    # the kernels' cents are the FP64 cents (tests/test_qoe_statistics.py): only FP32 summation differs
    np.testing.assert_allclose(got["Score"].cpu().numpy(), want, atol=1e-5, rtol=0)
    assert np.abs(got["Score"].cpu().numpy() - want).mean() < 2e-3
    np.testing.assert_allclose(got["Average QoE"].cpu().numpy(), all_qoe.mean(axis=1), atol=2e-4)
    idx, _ = scorer.best(5)
    assert set(idx.cpu().tolist()) <= set(np.argsort(-want)[:12].tolist())


@pytest.mark.parametrize("autoreset,steps", [(False, 20), (True, 47), (True, 1)])
def test_fused_rollout_equals_stepping_custom(autoreset, steps):
    """mbe_rollout on the fork's own scenario (one launch, state on chip between the steps) against
    the same number of mbe_step + mbe_accumulate_qoe calls: final state, score statistics and the
    per-step series must be bit-identical (the stepping path is pinned to the reference above)."""
    from mobile_env_gan_b200.scenarios import MComCustom
    from mobile_env_gan_b200.scoring import LayoutScorer

    E = 4096
    cfg = {"num_envs": E, "autoreset": autoreset}
    a, b = MComCustom(config=dict(cfg)), MComCustom(config=dict(cfg))
    sa, sb = LayoutScorer(a, 0.1), LayoutScorer(b, 0.1)
    a.reset(), b.reset()
    a.step(0, 0), b.step(0, 0)  # start mid-episode
    sa.acc.fill_(0.5), sb.acc.fill_(0.5)  # existing statistics are continued
    before = a.launch_count
    series = sa.run_episode(steps, record=("pos", "assoc", "rate", "utility"))
    assert a.launch_count - before == 1
    for k in range(steps):
        b.step(0, k)
        sb.update()
        torch.cuda.synchronize()
        assert torch.equal(series["assoc"][k], b.assoc), k
        assert torch.equal(series["rate"][k], b.rate), k
        assert torch.equal(series["utility"][k], b.utility_scaled), k
        if not (autoreset and bool(b.done.any())):  # on a reset step b.pos already holds the new episode
            assert torch.equal(series["pos"][k], b.pos), k
    for name in ("pos", "wp", "t", "episode", "assoc", "rate", "utility_scaled", "metrics", "bs_xy", "nbs", "done"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name
    assert torch.equal(sa.acc, sb.acc)


def test_rollout_positions_on_reset_steps_are_the_moved_ones():
    """The position series holds the positions after the move (what the reference dumps,
    base.py:232-233, 298-404) also on the step that ends an episode and auto-resets."""
    from mobile_env_gan_b200.scenarios import MComCustom

    E = 2048
    a = MComCustom(config={"num_envs": E, "autoreset": True})
    b = MComCustom(config={"num_envs": E, "autoreset": False})
    a.reset(), b.reset()
    series = a.rollout(20, record=("pos",))
    for k in range(20):
        b.step(0, k)
    assert bool(b.done.all()) and torch.equal(series["pos"][19], b.pos)
    assert int(a.episode.min()) == 1 and int(a.t.max()) == 0


@pytest.mark.parametrize("size,autoreset,steps", [("small", True, 47), ("medium", True, 47), ("medium", False, 20)])
def test_fused_rollout_equals_stepping_scenario_shapes(size, autoreset, steps):
    """The fused episode for the scenario shapes in FORK mode (one BS layout shared by all envs:
    step_tpe_fork_kernel<U,B,ROLLOUT,SHARED>): one launch against the same number of mbe_step +
    mbe_accumulate_qoe calls on the warp-segment kernel -- final state, score statistics and per-step
    series bit-identical."""
    from mobile_env_gan_b200.scenarios import MComMedium, MComSmall
    from mobile_env_gan_b200.scoring import LayoutScorer

    cls = {"small": MComSmall, "medium": MComMedium}[size]
    E = 2048
    cfg = {"num_envs": E, "autoreset": autoreset, "mode": "fork", "ue": {"velocity": 7.5}}
    a, b = cls(config=dict(cfg)), cls(config=dict(cfg))
    sa, sb = LayoutScorer(a, 0.1), LayoutScorer(b, 0.1)
    a.reset(), b.reset()
    a.step(0, 0), b.step(0, 0)  # start mid-episode
    sa.acc.fill_(0.25), sb.acc.fill_(0.25)
    before = a.launch_count
    series = sa.run_episode(steps, record=("pos", "wp", "assoc", "rate", "utility"))
    assert a.launch_count - before == 1
    for k in range(steps):
        b.step(0, k)
        sb.update()
        torch.cuda.synchronize()
        assert torch.equal(series["assoc"][k], b.assoc), k
        assert torch.equal(series["rate"][k], b.rate), k
        assert torch.equal(series["utility"][k], b.utility_scaled), k
        if not (autoreset and bool(b.done.any())):
            assert torch.equal(series["pos"][k], b.pos) and torch.equal(series["wp"][k], b.wp), k
    for name in ("pos", "wp", "t", "episode", "assoc", "rate", "utility_scaled", "metrics", "done"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name
    assert torch.equal(sa.acc, sb.acc)
    assert int(b.assoc.max()) >= 0 and len(torch.unique(b.assoc)) > 2  # several BSs really serve UEs


def test_rollout_other_shapes_run_as_step_sequence():
    """Shapes without the fused kernel: same API, same results, one launch per step."""
    from mobile_env_gan_b200.scoring import LayoutScorer

    MComCore, BaseStation, UserEquipment = _mods()
    a = make_env(SCENARIOS["small"][0], 5, {"num_envs": 300})
    b = make_env(SCENARIOS["small"][0], 5, {"num_envs": 300})
    sa, sb = LayoutScorer(a), LayoutScorer(b)
    a.reset(), b.reset()
    series = sa.run_episode(12, record=("pos", "rate", "assoc", "utility"))
    for k in range(12):
        b.step(0, k)
        sb.update()
        assert torch.equal(series["pos"][k], b.pos) and torch.equal(series["rate"][k], b.rate)
        assert torch.equal(series["assoc"][k], b.assoc) and torch.equal(series["utility"][k], b.utility_scaled)
    assert torch.equal(sa.acc, sb.acc) and torch.equal(a.pos, b.pos) and torch.equal(a.t, b.t)
    import mobile_env_gan_b200 as mbe
    from mobile_env_gan_b200._lib import MbeError

    g = mbe.make("mobile-small-central-v0", num_envs=64)
    g.reset()
    with pytest.raises(MbeError):
        g.rollout(3)


def test_errors_are_loud():
    MComCore, BaseStation, UserEquipment = _mods()
    from mobile_env_gan_b200._lib import MbeError

    with pytest.raises(MbeError):
        make_env(SCENARIOS["small"][0], 2000, {"num_envs": 4})  # U > 1024 has no kernel
    with pytest.raises(MbeError):  # the block-per-env kernel measures distances in exact FP32: d2 < 2^24
        wide_env("wide_rf", "gym", "central", 4, autoreset=False,
                 extra={"width": 5000, "height": 5000, "movement_params": {"width": 5000, "height": 5000}})
    wide, _, _ = wide_env("wide_rf", "gym", "central", 4, autoreset=False)
    with pytest.raises(MbeError):
        wide.step_window(1, 2)  # windows start at a multiple of 32 envs
    env = make_env(SCENARIOS["small"][0], 5, {"num_envs": 4})
    with pytest.raises(RuntimeError):
        env.step(0, 0)  # reset() first


# ------------------------------------------- block-per-env kernel: every entry point of the ABI
@pytest.mark.parametrize("name,mode,handler", [("wide_pf", "gym", "ma"), ("wide_rf", "gym", "central"),
                                               ("synthetic", "gym", "ma"), ("wide_rf", "fork", "central")])
def test_wide_split_phases_observe_and_windows_equal_the_fused_step(name, mode, handler):
    """mbe_stage (one launch per phase), mbe_observe and mbe_step_window on the block-per-env kernel
    reproduce its fused step bit for bit, over an episode end with autoreset."""
    from mobile_env_gan_b200 import _lib

    E = 34 if name == "synthetic" else 40
    fused, B, U = wide_env(name, mode, handler, E, autoreset=True)
    split, _, _ = wide_env(name, mode, handler, E, autoreset=True)
    wins, _, _ = wide_env(name, mode, handler, E, autoreset=True)
    for env in (fused, split, wins):
        env.reset()
    gym = mode == "gym"
    names = ["pos", "wp", "t", "episode", "rate", "utility_scaled", "metrics", "done"] + (
        ["conn", "obs", "reward"] if gym else ["assoc"])
    order = ([_lib.PHASE_PRE, _lib.PHASE_MOVE, _lib.PHASE_CLOCK, _lib.PHASE_POST] if gym else
             [_lib.PHASE_MOVE, _lib.PHASE_PRE, _lib.PHASE_CLOCK])
    rng = np.random.default_rng(5)
    side = torch.cuda.Stream()
    for k in range(10):
        if gym:
            acts = torch.from_numpy(rng.integers(0, B + 1, size=(E, U)).astype(np.int32)).cuda()
            fused.step(acts)
            split.actions.copy_(acts)
            wins.actions.copy_(acts)
        else:
            fused.step(0, k)
        for phase in order:
            split.stage(phase)
        torch.cuda.synchronize()
        wins.step_window(32, E - 32, stream=side)
        wins.step_window(0, 32)
        torch.cuda.synchronize()
        for n in names:
            assert torch.equal(getattr(split, n), getattr(fused, n)), (n, k)
            assert torch.equal(getattr(wins, n), getattr(fused, n)), (n, k)
        if gym:
            before = fused.obs.clone()
            fused.obs.zero_()
            fused.observe()
            assert torch.equal(fused.obs, before), k


def test_wide_debug_snr_matches_oracle():
    env, B, U = wide_env("wide_rf", "gym", "central", 8, autoreset=False)
    mir = Mirror(env)
    env.reset(), mir.reset()
    snr = env.enable_debug_snr()
    from oracle import mbe_oracle as orc

    for k in range(3):
        acts = np.zeros((8, U), dtype=np.int32)
        want, _ = orc.batch_snr(mir.p, mir.pos, mir.bs)
        env.step(torch.from_numpy(acts).cuda())
        mir.step_gym(acts)
        got = snr.cpu().numpy().astype(np.float64)
        fin = want < 3e38
        close(got[fin], want[fin], f"snr step {k}")


def test_full_size_synthetic_matches_compiled_oracle():
    """BASELINE configs[4] at FULL size: 64 BS x 512 UE, ProportionalFair, 16,384 envs (8.4 M UEs, 537 M
    links per step) against the compiled restatement, two steps -- connection sets, positions, done and
    FP64 rates exact, utilities / reward / observations 1e-5 (compared in env slices)."""
    CEnvBatch = _compiled_oracle()
    E = 16384
    env, B, U = wide_env("synthetic", "gym", "central", E, autoreset=False)
    mir = Mirror(env)
    env.reset()
    mir._reinit(np.ones(E, dtype=bool))
    c = CEnvBatch(mir.p, mir.bs, E, U, handler="central", pinned_tables=True)
    c.reset(mir.pos)
    rng = np.random.default_rng(4)
    for k in range(2):
        acts = rng.integers(0, B + 1, size=(E, U)).astype(np.int32)
        mir.t = c.t.astype(np.int64)
        c.step_gym(acts, mir.new_wp())
        obs, rew, _, trunc, _ = env.step(torch.from_numpy(acts).to(env.device))
        assert np.array_equal(env.pos.cpu().numpy(), c.pos), k
        assert np.array_equal(trunc.cpu().numpy(), c.done.astype(bool)), k
        close(rew.cpu(), c.reward, f"reward {k}")
        for lo in range(0, E, 1024):
            sl = slice(lo, lo + 1024)
            assert np.array_equal(conn_bool_from_words(env.conn[sl].cpu().numpy(), B), c.conn[sl].astype(bool)), (k, lo)
            _rates_bit_exact(env.rate[sl].cpu().numpy(), c.rate[sl], f"rate step {k} envs {lo}..")  # 8.4 M FP64 rates
            close(env.utility_scaled[sl].cpu(), c.util[sl], f"utility {k}")
            close(obs[sl].cpu().numpy().reshape(1024, U, -1), c.obs[sl], f"obs {k}")


def test_full_size_large_central_matches_compiled_oracle():
    """BASELINE configs[3] at FULL size: mobile-large-central-v0 (13 BS x 30 UE) on 262,144 envs, five
    Philox-driven steps against the compiled restatement."""
    import mobile_env_gan_b200 as mbe

    CEnvBatch = _compiled_oracle()
    E = 262144
    env = mbe.make("mobile-large-central-v0", num_envs=E)
    mir = Mirror(env)
    env.reset()
    mir._reinit(np.ones(E, dtype=bool))
    U, B = mir.U, mir.B
    c = CEnvBatch(mir.p, mir.bs, E, U, handler="central", pinned_tables=True)
    c.reset(mir.pos)
    rng = np.random.default_rng(9)
    for k in range(5):
        acts = rng.integers(0, B + 1, size=(E, U)).astype(np.int32)
        mir.t = c.t.astype(np.int64)
        c.step_gym(acts, mir.new_wp())
        obs, rew, _, trunc, _ = env.step(torch.from_numpy(acts).to(env.device))
        assert np.array_equal(conn_bool_from_words(env.conn.cpu().numpy(), B), c.conn.astype(bool)), k
        assert np.array_equal(env.pos.cpu().numpy(), c.pos), k
        assert np.array_equal(trunc.cpu().numpy(), c.done.astype(bool)), k
        _rates_bit_exact(env.rate.cpu().numpy(), c.rate, f"rate step {k}")
        close(env.utility_scaled.cpu(), c.util, f"utility {k}")
        close(rew.cpu(), c.reward, f"reward {k}")
        for lo in range(0, E, 32768):
            close(obs[lo:lo + 32768].cpu().numpy().reshape(32768, U, -1), c.obs[lo:lo + 32768], f"obs {k}")
