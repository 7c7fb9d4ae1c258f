"""Map-panel frames (mbe_render, DESIGN.md section 9): the CUDA kernel against the numpy restatement
oracle/render_ref.py byte for byte, series frames against stepping, the gymnasium render surface, and
the integer predicates of the specification on the CPU."""
import ctypes as C

import numpy as np
import pytest

from oracle import render_ref
from mobile_env_gan_b200 import render as R

SIZES = [(64, 64), (200, 200), (96, 160), (512, 512)]


def _make(bs_xy, nue, config, bs_over=None):
    from mobile_env_gan_b200.core.base import MComCore
    from mobile_env_gan_b200.core.entities import BaseStation, UserEquipment
    from mobile_env_gan_b200.core.util import deep_dict_merge

    cfg = deep_dict_merge(MComCore.default_config(), config)
    stations = []
    for i, xy in enumerate(bs_xy):
        kw = dict(cfg["bs"])
        kw.update((bs_over or {}).get(i, {}))
        stations.append(BaseStation(i, tuple(xy), **kw))
    users = [UserEquipment(i, **cfg["ue"]) for i in range(nue)]
    return MComCore(stations, users, config)


TWO_CLASS_BS = [(40, 40), (160, 50), (100, 150), (30, 170)]


def two_class_plan_parts():
    """A layout whose BSs 1 and 3 transmit at lower power: two BS classes of different d2max."""
    from mobile_env_gan_b200.core.base import MComCore
    from mobile_env_gan_b200.core.entities import BaseStation, UserEquipment

    cfg = MComCore.seeding(MComCore.default_config())
    stations = [BaseStation(i, xy, **dict(cfg["bs"], **({"tx": 25} if i % 2 else {})))
                for i, xy in enumerate(TWO_CLASS_BS)]
    users = [UserEquipment(i, **cfg["ue"]) for i in range(9)]
    return stations, users, cfg


# ------------------------------------------------------------------------------------- CPU ----
def test_coverage_is_the_connectable_set_on_a_one_to_one_frame():
    from mobile_env_gan_b200.core.base import MComCore

    stations, users, cfg = two_class_plan_parts()
    plan = MComCore.build_plan(stations, users, cfg)
    d2 = render_ref.link_d2max(plan)
    assert len(set(d2.tolist())) == 2 and d2.min() >= 0
    Wm, Hm = int(cfg["width"]), int(cfg["height"])
    xs, ys = render_ref.sample_points(Hm, Wm, Wm, Hm)
    assert np.array_equal(xs, np.arange(Wm)) and np.array_equal(ys, np.arange(Hm)[::-1])
    cnt = render_ref.coverage_counts(xs, ys, TWO_CLASS_BS, d2)
    brute = np.zeros((Hm, Wm), dtype=np.int64)  # row 0 is y = Hm - 1
    for (bx, by), dm in zip(TWO_CLASS_BS, d2):
        for y in range(Hm):
            for x in range(Wm):
                brute[Hm - 1 - y, x] += (x - bx) ** 2 + (y - by) ** 2 <= dm
    assert np.array_equal(cnt, brute)
    frame = render_ref.render_frame(cfg["width"], cfg["height"], TWO_CLASS_BS, d2, np.zeros((0, 2)),
                                    np.zeros((0, 4), bool), np.zeros(0, np.float32), size=(Hm, Wm), bs_half=0)
    tint = np.minimum(brute, 3)
    bs_pix = np.zeros_like(brute, dtype=bool)
    for bx, by in TWO_CLASS_BS:
        bs_pix[Hm - 1 - by, bx] = True
    assert np.array_equal(frame[~bs_pix], R.PALETTE[tint][~bs_pix])


def _seg_dist2(px, py, ax, ay, bx, by):
    p, a, b = (np.array(v, dtype=np.float64) for v in ((px, py), (ax, ay), (bx, by)))
    d = b - a
    L = d @ d
    t = 0.0 if L == 0 else np.clip((p - a) @ d / L, 0.0, 1.0)
    q = a + t * d - p
    return q @ q


def test_segment_predicate_matches_float_distance():
    rng = np.random.default_rng(7)
    checked = 0
    for _ in range(20000):
        px, py, ax, ay, bx, by = rng.integers(0, 60, size=6)
        w = int(rng.integers(0, 9))
        d2 = _seg_dist2(px, py, ax, ay, bx, by)
        if abs(4 * d2 - w * w) < 1e-6:  # ties: exactly on the boundary, decided by the integer form only
            continue
        assert bool(render_ref.on_segment(px, py, ax, ay, bx, by, w)) == (4 * d2 < w * w), (px, py, ax, ay, bx, by, w)
        checked += 1
    assert checked > 19000
    py, px = np.mgrid[0:20, 0:20]
    horiz = render_ref.on_segment(px, py, 2, 10, 17, 10, 3)  # width 3: rows 9..11 (d = 1), ends rounded
    assert horiz[10, 2:18].all() and horiz[9, 2:18].all() and not horiz[8].any() and not horiz[12].any()
    assert horiz[10, 1] and not horiz[10, 0] and horiz[10, 18] and horiz[9, 1] and not horiz[9, 0]  # 4*2 <= 9 < 4*5
    vert = render_ref.on_segment(px, py, 5, 3, 5, 16, 1)  # width 1: exactly the column
    assert np.array_equal(vert, (px == 5) & (py >= 3) & (py <= 16))
    diag = render_ref.on_segment(px, py, 0, 0, 19, 19, 1)  # width 1: the diagonal itself
    assert np.array_equal(diag, px == py)
    dot = render_ref.on_segment(px, py, 7, 7, 7, 7, 4)  # degenerate segment: a disc of radius 2
    assert np.array_equal(dot, (px - 7) ** 2 + (py - 7) ** 2 <= 4)


def test_utility_ramp_index_at_bucket_boundaries():
    assert render_ref.R.ramp_index([-1.0, 0.0, 1.0]).tolist() == [0, 128, 255]
    f32 = np.float32
    bounds = np.array([k / 128.0 - 1.0 for k in range(1, 256)], dtype=np.float32)
    vals = np.concatenate([bounds, np.nextafter(bounds, f32(-2)), np.nextafter(bounds, f32(2)),
                           np.array([-1.5, -1.0, np.nextafter(f32(-1), f32(0)), 1.0, np.nextafter(f32(1), f32(0)), 2.0],
                                    dtype=np.float32)])
    # independent statement: u + 1 is exact in float64 and rounded once to float32, * 128 is exact
    v = np.floor(np.float32(vals.astype(np.float64) + 1.0).astype(np.float64) * 128.0)
    want = np.clip(v, 0, 255).astype(np.int64)
    assert np.array_equal(R.ramp_index(vals), want)
    assert R.ramp_index(bounds).tolist() == list(range(1, 256))
    assert R.ramp_index(np.nextafter(f32(-1 + 1 / 128), f32(-2))) == 0
    assert R.PALETTE.shape == (R.PALETTE_SIZE, 3) and R.PALETTE.dtype == np.uint8


def test_render_style_carries_the_palette():
    st = R.style((96, 160))
    assert (st.height, st.width, st.ue_radius, st.bs_half, st.line_width) == (96, 160, R.UE_RADIUS, R.BS_HALF,
                                                                            R.LINE_WIDTH)
    assert bytes(st.palette) == R.PALETTE.tobytes()
    from mobile_env_gan_b200 import _lib

    assert C.sizeof(_lib.RenderStyle) == 5 * 4 + 3 * _lib.RENDER_PALETTE + 2


# ------------------------------------------------------------------------------------- GPU ----
def _gym_stepped(env, steps=3, seed=0):
    import torch

    rng = np.random.default_rng(seed)
    env.reset()
    for _ in range(steps):
        acts = rng.integers(0, env.NUM_STATIONS + 1, size=(env.num_envs, env.NUM_USERS)).astype(np.int32)
        env.step(torch.from_numpy(acts).to(env.device))
    return env


def _expected(env, ids, size, series=None, step=0):
    """Frames of env ids from host copies of the state (or of one step of a series)."""
    bs = env.bs_xy.cpu().numpy()
    nbs = None if env.nbs is None else env.nbs.cpu().numpy()
    if series is None:
        pos, util = env.pos.cpu().numpy(), env.utility_scaled.cpu().numpy()
        conn = None if env.conn is None else env.conn.cpu().numpy().reshape(env.num_envs, env.NUM_USERS, -1)
        assoc = None if env.assoc is None else env.assoc.cpu().numpy()
    else:
        pos, util = series["pos"][step].cpu().numpy(), series["utility"][step].cpu().numpy()
        conn, assoc = None, series["assoc"][step].cpu().numpy()
    out = []
    for e in ids:
        out.append(render_ref.render_env_state(
            env.plan, env.width, env.height, bs[e] if bs.ndim == 3 else bs, None if nbs is None else nbs[e], pos[e],
            None if conn is None else conn[e], None if assoc is None else assoc[e], util[e], size=size))
    return np.stack(out)


def _case(name):
    import mobile_env_gan_b200 as mbe
    from mobile_env_gan_b200.scenarios.custom import MComCustom

    if name in ("small-central", "medium-ma", "large-central", "large-ma"):
        size, h = name.split("-")
        return _gym_stepped(mbe.make(f"mobile-{size}-{h}-v0", num_envs=40, device="cuda:0"))
    if name == "custom-fork":
        env = MComCustom(config={"num_envs": 64})
        env.reset()
        for s in range(4):
            env.step(0, s)
        assert int(env.nbs.min()) < env.plan.num_bs
        return env
    if name == "two-class":
        stations, users, cfg = two_class_plan_parts()
        from mobile_env_gan_b200.core.base import MComCore

        env = MComCore(stations, users, {"num_envs": 40, "mode": "gym", "handler": "central"})
        assert env.plan.num_bs_classes == 2
        return _gym_stepped(env)
    if name == "wide-70x40":
        rng = np.random.default_rng(40 * 1000 + 70)
        bs = rng.integers(0, 200, size=(40, 2)).tolist()
        env = _make(bs, 70, {"num_envs": 12, "mode": "gym", "handler": "central", "ue": {"velocity": 9},
                             "movement_params": {"reset_rng_episode": False}})
        assert env.conn.dim() == 3 and env.conn.shape[2] == 2
        return _gym_stepped(env, steps=4)
    raise KeyError(name)


CASES = ["small-central", "medium-ma", "large-central", "large-ma", "custom-fork", "two-class", "wide-70x40"]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_kernel_frames_equal_the_restatement(case):
    env = _case(case)
    E = env.num_envs
    ids = [E - 1, E - 3, 5, E - 3, 1, 0]  # reversed subset with one duplicate
    if case in ("small-central", "two-class"):  # several UEs must hold several connections
        conn = env.conn.cpu().numpy().astype(np.int64) & 0xFFFFFFFF
        assert max(bin(int(c)).count("1") for c in conn.reshape(-1)) >= 2
    for size in SIZES:
        got = env.render_frames(ids, size=size).cpu().numpy()
        assert got.shape == (len(ids), size[0], size[1], 3) and got.dtype == np.uint8
        want = _expected(env, ids, size)
        for k in range(len(ids)):
            assert np.array_equal(got[k], want[k]), (case, size, k, int((got[k] != want[k]).any(-1).sum()))
    full = env.render_frames().cpu().numpy()  # envs=None: all envs in order
    assert full.shape[0] == E and np.array_equal(full[1], _expected(env, [1], None)[0])


@pytest.mark.gpu
def test_ramp_boundaries_and_line_widths_on_the_gpu():
    import torch
    from mobile_env_gan_b200 import _lib

    env = _case("custom-fork")
    f32 = np.float32
    bounds = np.array([k / 128.0 - 1.0 for k in range(1, 256)], dtype=np.float32)
    vals = np.concatenate([bounds, np.nextafter(bounds, f32(-2)), np.nextafter(bounds, f32(2))])
    u = np.resize(vals, env.utility_scaled.numel()).reshape(env.utility_scaled.shape)
    env.utility_scaled.copy_(torch.from_numpy(u))
    ids = list(range(env.num_envs))
    assert np.array_equal(env.render_frames(ids, size=(64, 64)).cpu().numpy(), _expected(env, ids, (64, 64)))
    # other entity sizes through the C entry (render_frames uses the default style)
    for r, s, w in ((0, 0, 0), (6, 2, 4), (1, 9, 7)):
        st = R.style((96, 128), ue_radius=r, bs_half=s, line_width=w)
        out = torch.empty((1, 4, 96, 128, 3), dtype=torch.uint8, device=env.device)
        ids_t = torch.tensor([3, 2, 1, 0], dtype=torch.int32, device=env.device)
        _lib.check(env._lib.mbe_render(env._handle, C.c_void_p(ids_t.data_ptr()), 4, None, 1, C.byref(st),
                                       C.c_void_p(out.data_ptr()), env._stream()))
        bs, nbs = env.bs_xy.cpu().numpy(), env.nbs.cpu().numpy()
        pos, assoc, ut = env.pos.cpu().numpy(), env.assoc.cpu().numpy(), env.utility_scaled.cpu().numpy()
        for k, e in enumerate([3, 2, 1, 0]):
            nb = int(nbs[e])
            conn = np.zeros((7, nb), bool)
            for uu in range(7):
                if 0 <= assoc[e, uu] < nb:
                    conn[uu, assoc[e, uu]] = True
            want = render_ref.render_frame(env.width, env.height, bs[e, :nb], render_ref.link_d2max(env.plan)[:nb],
                                           pos[e], conn, ut[e], size=(96, 128), ue_radius=r, bs_half=s, line_width=w)
            assert np.array_equal(out[0, k].cpu().numpy(), want), (r, s, w, e)


@pytest.mark.gpu
def test_out_of_range_env_ids_give_background_frames_in_the_kernel():
    import torch
    from mobile_env_gan_b200 import _lib

    env = _case("small-central")
    st = R.style((32, 64))
    ids = torch.tensor([-1, env.num_envs, 2], dtype=torch.int32, device=env.device)
    out = torch.zeros((1, 3, 32, 64, 3), dtype=torch.uint8, device=env.device)
    _lib.check(env._lib.mbe_render(env._handle, C.c_void_p(ids.data_ptr()), 3, None, 1, C.byref(st),
                                   C.c_void_p(out.data_ptr()), env._stream()))
    o = out.cpu().numpy()
    assert (o[0, :2] == R.PALETTE[R.BACKGROUND]).all()
    assert np.array_equal(o[0, 2], _expected(env, [2], (32, 64))[0])


@pytest.mark.gpu
def test_series_frames_equal_frames_after_each_step():
    from mobile_env_gan_b200.scenarios.custom import MComCustom

    a, b = MComCustom(config={"num_envs": 256}), MComCustom(config={"num_envs": 256})
    a.reset(), b.reset()
    n0 = a.launch_count
    series = a.rollout(20, record=("pos", "assoc", "utility"))
    n1 = a.launch_count
    frames = a.render_frames(size=(128, 128), series=series)
    assert a.launch_count == n1 + 1 and n1 > n0
    assert frames.shape == (20, 256, 128, 128, 3)
    ids = [255, 7, 0]
    sub = a.render_frames(ids, size=(96, 160), series=series)
    for s in range(20):
        b.step(0, s)
        assert np.array_equal(frames[s].cpu().numpy(), b.render_frames(size=(128, 128)).cpu().numpy()), s
        if s in (0, 19):
            assert np.array_equal(sub[s].cpu().numpy(), _expected(a, ids, (96, 160), series, s))


@pytest.mark.gpu
def test_render_surface():
    import mobile_env_gan_b200 as mbe

    env = mbe.make("mobile-medium-central-v0", num_envs=8, device="cuda:0", render_mode="rgb_array")
    _gym_stepped(env, steps=2)
    img = env.render()
    assert isinstance(img, np.ndarray) and img.shape == (*R.DEFAULT_SIZE, 3) and img.dtype == np.uint8
    assert np.array_equal(img, env.render_frames([0])[0].cpu().numpy())
    assert mbe.make("mobile-small-central-v0", num_envs=2, device="cuda:0").render() is None
    human = mbe.make("mobile-small-central-v0", num_envs=2, device="cuda:0", render_mode="human")
    with pytest.raises(NotImplementedError, match="display"):
        human.render()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["medium-ma", "custom-fork"])
def test_rendering_changes_nothing(case):
    import torch

    a, b = _case(case), _case(case)
    sd = a.state_dict()
    n = a.launch_count
    a.render_frames([0])
    assert a.launch_count == n + 1
    a.render_frames(size=(64, 64))
    assert a.launch_count == n + 2
    after = a.state_dict()
    assert all(torch.equal(sd[k], after[k]) for k in sd)
    if a.plan.mode == 1:
        acts = torch.ones((a.num_envs, a.NUM_USERS), dtype=torch.int32, device=a.device)
        oa, ra, _, ta, _ = a.step(acts)
        ob, rb, _, tb, _ = b.step(acts.clone())
        assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(ta, tb)
    else:
        a.step(0, 9), b.step(0, 9)
    for k, v in a.state_dict().items():
        assert torch.equal(v, b.state_dict()[k]), k


@pytest.mark.gpu
def test_render_errors_are_loud():
    from mobile_env_gan_b200 import _lib

    gym = _case("small-central")
    with pytest.raises(_lib.MbeError, match="multiple of 4"):
        gym.render_frames([0], size=(64, 66))
    with pytest.raises(_lib.MbeError, match="out of range"):
        gym.render_frames([0], size=(4, 64))
    with pytest.raises(IndexError):
        gym.render_frames([0, gym.num_envs])
    with pytest.raises(IndexError):
        gym.render_frames([-1])
    fork = _case("custom-fork")
    series = fork.rollout(2, record=("pos", "assoc", "utility"))
    with pytest.raises(_lib.MbeError, match="FORK"):
        gym.render_frames([0], series=series)
    with pytest.raises(_lib.MbeError, match="needs pos"):
        fork.render_frames([0], series={"assoc": series["assoc"], "utility": series["utility"]})
