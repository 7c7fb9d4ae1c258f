"""Layout maps (``mbe_layout_map``, DESIGN.md section 10.2): coverage, serving BS and QoE cent per grid point and
the map-wide statistics, against the numpy restatement ``oracle/map_ref.py`` with ``==``; the serving BS, rate
and cent against what the step's PRE phase computes for UEs placed on grid points; no side effects; the
error cases of the entry."""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import pytest

from oracle import map_ref, qoe_ref

from mobile_env_gan_b200 import _lib


def _brute(width, height, stride, bs, nb, d2max, cent_tabs, threshold):
    """The specification point by point in Python integers."""
    xs = range(0, math.ceil(width), stride)
    ys = range(0, math.ceil(height), stride)
    cov, srv, qoe = [], [], []
    for y in ys:
        for x in xs:
            c, best, bd = 0, -1, None
            for b in range(max(0, min(nb, len(bs)))):
                d2 = (x - bs[b][0]) ** 2 + (y - bs[b][1]) ** 2
                if d2 <= d2max[b]:
                    c += 1
                    if bd is None or d2 < bd:
                        best, bd = b, d2
            cov.append(c)
            srv.append(best)
            qoe.append(-100 if best < 0 else int(cent_tabs[best][bd]))
    k = np.array(qoe)
    low = sum(1 for v in qoe if float(np.float32(v / 100)) < float(np.float32(threshold)))
    stats = [len(qoe), sum(c >= 1 for c in cov), sum(c >= 2 for c in cov), int(k.sum()), int((k * k).sum()), low]
    area = [sum(s == b for s in srv) for b in range(len(bs))]
    shape = (len(ys), len(xs))
    return np.array(cov).reshape(shape), np.array(srv).reshape(shape), k.reshape(shape), stats, area


# ------------------------------------------------------------------------------------------- CPU --
HAND_MADE = {
    # BS on grid points (d2 = 0), two BSs at the same distance from many points (ties), a far BS
    "ties": (50, 40, 1, [(10, 10), (30, 10), (20, 30), (-300, 5)], 4, [100, 100, 49, 10]),
    "dead-slots": (50, 40, 3, [(10, 10), (30, 10), (20, 30), (25, 20)], 2, [400, 400, 400, 400]),
    "out-of-range": (30, 30, 2, [(100, 100), (-50, 0)], 2, [25, 25]),
    "never-connectable": (20, 20, 1, [(5, 5), (15, 15)], 2, [-1, 36]),
    "non-integer-map": (40.5, 20.25, 4, [(0, 0), (40, 20), (8, 12)], 3, [200, 300, 64]),
    "stride-not-dividing": (37, 23, 7, [(14, 7), (35, 21)], 2, [150, 150]),
}


@pytest.mark.parametrize("case", sorted(HAND_MADE))
@pytest.mark.parametrize("threshold", [0.0, 0.1, 0.5])
def test_restatement_equals_the_specification_point_by_point(case, threshold):
    width, height, stride, bs, nb, d2max = HAND_MADE[case]
    rng = np.random.default_rng(7)
    tabs = [rng.integers(-100, 101, size=max(d, 0) + 1) for d in d2max]
    xs, ys = map_ref.grid(width, height, stride)
    assert xs[-1] <= math.ceil(width) - 1 < xs[-1] + stride and ys[-1] <= math.ceil(height) - 1 < ys[-1] + stride
    cov, srv, k, stats, area = map_ref.env_map(xs, ys, bs, nb, d2max, tabs, threshold)
    bcov, bsrv, bk, bstats, barea = _brute(width, height, stride, bs, nb, d2max, tabs, threshold)
    assert np.array_equal(cov, bcov) and np.array_equal(srv, bsrv) and np.array_equal(k, bk)
    assert stats.tolist() == bstats and area.tolist() == barea
    assert cov.dtype == np.uint8 and srv.dtype == np.int8 and k.dtype == np.int8
    if case == "ties":
        assert cov.max() >= 2 and (k[srv < 0] == -100).all() and (srv < 0).any()
        assert srv[10, 20] == 0  # equidistant from slots 0 and 1: the lower slot serves
    if case == "dead-slots":
        assert srv.max() <= 1 and area[2:].sum() == 0
    if case == "out-of-range":
        assert (cov == 0).all() and stats[1] == 0 and stats[3] == -100 * stats[0]


def test_grid_of_a_non_integer_map_is_the_range_of_the_ue_draws():
    xs, ys = map_ref.grid(200.5, 99.01, 1)
    assert xs[-1] == 200 and ys[-1] == 99  # int(u * 200.5) reaches 200, int(u * 99.01) reaches 99
    xs, ys = map_ref.grid(200, 200, 3)
    assert len(xs) == 67 and xs[-1] == 198


def test_k_low_is_the_low_qoe_test_at_every_cent_and_near_cent_threshold():
    ks = np.arange(-100, 101)
    thresholds = np.concatenate([qoe_ref.cent_thresholds(), qoe_ref.near_cents_and_ties(2),
                                 np.array([0.1, -0.1, 0.5, 2.0, -2.0], dtype=np.float32)])
    for t in thresholds:
        kl = map_ref.k_low(float(t))
        assert np.array_equal(ks < kl, qoe_ref.is_low(ks, float(t))), t
        # the library's loop: the smallest k with float32(k / 100) >= float32(threshold), else 101
        want = next((k for k in range(-100, 101) if np.float32(np.float64(k) / 100.0) >= np.float32(t)), 101)
        assert kl == want, t
    assert map_ref.k_low(0.1) == 10 and map_ref.k_low(0.0) == 0 and map_ref.k_low(-0.0) == 0
    assert map_ref.k_low(1.5) == 101 and map_ref.k_low(-1.5) == -100


def test_result_keys_follow_the_notebook_formula():
    k = np.array([-100, -100, 20, 35, 35, 100])
    stats = np.array([6, 4, 2, k.sum(), (k * k).sum(), 2])
    r = map_ref.result(stats)
    q = k / 100
    assert math.isclose(r["Average QoE"], q.mean(), abs_tol=1e-15)
    assert math.isclose(r["QoE Variance"], q.var(), abs_tol=1e-15)
    assert r["Low QoE Proportion"] == 2 / 6 and r["Coverage"] == 4 / 6 and r["Overlap"] == 2 / 6


def test_map_params_struct_size_matches_the_library():
    lib = _lib.load()
    assert lib.mbe_struct_size(7) == C.sizeof(_lib.MapParams) == 20
    assert lib.mbe_struct_size(8) == -1


# ------------------------------------------------------------------------------------------- GPU --
def _cent_tabs(plan, load, ue_class):
    """Per BS class: the cents per d2 of the link class (BS class, ue_class) at this load."""
    nuc = len(plan.ue_classes) if plan.ue_class is not None else 1
    tabs, d2max = [], []
    for c in range(plan.num_bs_classes):
        cl = plan.classes[c * nuc + ue_class]
        d = int(cl["d2max"])
        d2max.append(d)
        lut = np.asarray(cl["rate_lut"], dtype=np.float64)[: d + 1] if d >= 0 else np.zeros(0)
        tabs.append(map_ref.cents_of_rates(map_ref.shared_rate(lut, load), plan.utility))
    return tabs, d2max


def _expected(env, ids, stride=1, load=1, ue_class=0, threshold=0.0):
    p = env.plan
    E, B = env.num_envs, p.num_bs
    xs, ys = map_ref.grid(p.width, p.height, stride)
    tabs, d2max = _cent_tabs(p, load, ue_class)
    bcls = p.bs_class if p.bs_class is not None else np.zeros(B, dtype=np.uint8)
    slot_d2 = [d2max[c] for c in bcls]
    slot_tab = [tabs[c] for c in bcls]
    bs = env.bs_xy.cpu().numpy()
    nbs = env.nbs.cpu().numpy() if env.nbs is not None else None
    out = []
    for e in ids:
        if not 0 <= e < E:
            out.append(map_ref.empty_map(xs, ys, B))
            continue
        layout = bs[e] if bs.ndim == 3 else bs
        out.append(map_ref.env_map(xs, ys, layout, B if nbs is None else nbs[e], slot_d2, slot_tab, threshold))
    return [np.stack(v) for v in zip(*out)]


def _check(env, ids=None, **kw):
    """layout_map of ids (None: all envs) equals the restatement in every output."""
    n0 = env.launch_count
    m = env.layout_map(ids, **kw)
    assert env.launch_count == n0 + 2
    ids_l = list(range(env.num_envs)) if ids is None else [int(i) for i in ids]
    cov, srv, k, stats, area = _expected(env, ids_l, **kw)
    got = [m.coverage, m.serving, m.qoe, m.stats, m.area]
    for name, g, w in zip(("coverage", "serving", "qoe", "stats", "area"), got, (cov, srv, k, stats, area)):
        g = g.cpu().numpy()
        assert g.shape == w.shape, (name, g.shape, w.shape)
        bad = np.argwhere(g != w)
        assert bad.size == 0, (name, kw, bad[:3].tolist(), g[tuple(bad[0])], w[tuple(bad[0])])
    r = m.result()
    want = map_ref.result(stats)
    for key, v in want.items():
        assert np.array_equal(r[key].cpu().numpy(), v, equal_nan=True), key
    return m


def _custom(E, **cfg):
    from mobile_env_gan_b200.scenarios import MComCustom

    env = MComCustom(config={"num_envs": E, **cfg})
    env.reset()
    return env


def _shared(bs_xy, nue, config, bs_over=None, ue_over=None):
    from mobile_env_gan_b200.core.base import MComCore
    from mobile_env_gan_b200.core.entities import BaseStation, UserEquipment
    from mobile_env_gan_b200.core.util import deep_dict_merge

    cfg = deep_dict_merge(MComCore.default_config(), config)
    stations = [BaseStation(i, tuple(xy), **dict(cfg["bs"], **(bs_over or {}).get(i, {}))) for i, xy in enumerate(bs_xy)]
    users = [UserEquipment(i, **dict(cfg["ue"], **(ue_over or {}).get(i, {}))) for i in range(nue)]
    env = MComCore(stations, users, config)
    env.reset()
    return env


GRID = [(1, 1, 0.0), (3, 7, 0.1), (7, 1, 0.5), (7, 7, 0.0), (3, 1, 0.5), (1, 7, 0.1)]  # (stride, load, threshold)


@pytest.mark.gpu
@pytest.mark.parametrize("E", [64, 1 << 16])
def test_custom_per_env_layouts_equal_the_restatement(E):
    env = _custom(E)
    assert int(env.nbs.min()) < env.plan.num_bs  # dead slots in play
    rng = np.random.default_rng(E)
    sample = [0, E - 1, 5, 5, -1, E, E + 100] + rng.integers(0, E, size=24).tolist()
    for stride, load, thr in GRID:
        _check(env, sample, stride=stride, load=load, threshold=thr)
    if E == 64:
        _check(env, None, stride=3, load=1, threshold=0.1)  # every env, envs=None
    else:  # statistics only over every env at a coarse stride
        m = env.layout_map(stride=7, maps=False)
        assert m.coverage is None
        ids = rng.integers(0, E, size=64).tolist()
        _, _, _, stats, area = _expected(env, ids, stride=7)
        assert np.array_equal(m.stats.cpu().numpy()[ids], stats) and np.array_equal(m.area.cpu().numpy()[ids], area)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["mobile-small-central-v0", "mobile-medium-ma-v0", "mobile-large-central-v0"])
def test_shared_scenario_layouts_equal_the_restatement(name):
    import mobile_env_gan_b200 as mbe

    env = mbe.make(name, num_envs=40, device="cuda:0")
    env.reset()
    U = env.plan.num_ues
    for stride, load, thr in GRID:
        _check(env, [0, 39, 3, 3, -5, 40], stride=stride, load=U if load == 7 else load, threshold=thr)


@pytest.mark.gpu
def test_two_bs_classes_and_a_second_ue_class():
    bs = [(40, 40), (160, 50), (100, 150), (30, 170), (100, 100)]
    env = _shared(bs, 6, {"num_envs": 8, "mode": "gym", "handler": "central"},
                  bs_over={1: {"tx": 25}, 3: {"tx": 25}}, ue_over={u: {"snr_tr": 2e-7} for u in (1, 4, 5)})
    p = env.plan
    assert p.num_bs_classes == 2 and len(p.ue_classes) == 2
    _, d0 = _cent_tabs(p, 1, 0)
    _, d1 = _cent_tabs(p, 1, 1)
    assert d0 != d1 and len(set(d0)) == 2
    for ue_class in (0, 1):
        for stride, load, thr in GRID:
            _check(env, [0, 7, 2, 2, 8], stride=stride, load=6 if load == 7 else load, ue_class=ue_class, threshold=thr)


class _TwoSlope:
    """A power_loss-only channel that is not affine in log-distance: the kernels read a log2 snr table."""

    @staticmethod
    def make():
        from mobile_env_gan_b200.core.channels import Channel

        class TwoSlope(Channel):
            def __init__(self, gamma1=2.0, gamma2=4.5, d_break=25.0, **kwargs):
                super().__init__(**kwargs)
                self.gamma1, self.gamma2, self.d_break = gamma1, gamma2, d_break

            def power_loss(self, bs, ue):
                dist = bs.point.distance(ue.point)
                if dist <= self.d_break:
                    return 10 * self.gamma1 * np.log10(4 * np.pi * dist * bs.frequency)
                return (10 * self.gamma1 * np.log10(4 * np.pi * self.d_break * bs.frequency)
                        + 10 * self.gamma2 * np.log10(dist / self.d_break))

        return TwoSlope


@pytest.mark.gpu
def test_two_slope_tabulated_channel():
    env = _shared([(60, 60), (140, 60), (60, 140), (140, 140)], 10,
                  {"num_envs": 16, "mode": "fork", "channel": _TwoSlope.make(), "ue": {"velocity": 8, "snr_tr": 0.1}})
    assert env.plan.classes[0].get("log2snr_lut") is not None
    for stride, load, thr in GRID:
        _check(env, [0, 15, 1, 1, 99], stride=stride, load=10 if load == 7 else load, threshold=thr)


@pytest.mark.gpu
def test_block_per_env_handle_70_ues_40_bs():
    rng = np.random.default_rng(40 * 1000 + 70)
    bs = rng.integers(0, 200, size=(40, 2)).tolist()
    env = _shared(bs, 70, {"num_envs": 12, "mode": "gym", "handler": "central", "ue": {"velocity": 9},
                           "movement_params": {"reset_rng_episode": False}})
    assert env.step_kernel_name == "step_big_kernel"
    for stride, load, thr in GRID:
        _check(env, [11, 0, 4, 4, 12, -1], stride=stride, load=70 if load == 7 else load, threshold=thr)


def _placed(env, points, per_env):
    """Puts the UEs of env e on grid point points[e] (all of them, or the first when per_env == 1)."""
    import torch

    pos = env.pos.cpu().numpy()
    pos[:, :per_env] = points[:, None, :]
    env.set_positions(torch.from_numpy(pos))
    env.stage(_lib.PHASE_PRE)


@pytest.mark.gpu
def test_one_ue_per_env_agrees_with_the_step():
    """FORK, generic kernel: a UE alone on grid point e of env e is served by the map's serving BS, at the
    load-1 rate, with the map's cent."""
    stride = 7
    env = _shared([(40, 40), (160, 50), (100, 150), (30, 170), (100, 100)], 1,
                  {"num_envs": 29 * 29, "mode": "fork", "generic_kernel": True, "ue": {"snr_tr": 2e-5}})
    assert env.step_kernel_name == "step_kernel"
    xs, ys = map_ref.grid(env.plan.width, env.plan.height, stride)
    X, Y = np.meshgrid(xs, ys)
    pts = np.stack([X.ravel(), Y.ravel()], axis=1)
    assert len(pts) == env.num_envs
    _placed(env, pts, 1)
    m = env.layout_map([0], stride=stride, load=1)
    srv, k = m.serving.cpu().numpy()[0].ravel(), m.qoe.cpu().numpy()[0].ravel()
    assoc, rate, util = env.assoc.cpu().numpy()[:, 0], env.rate.cpu().numpy()[:, 0], env.utility_scaled.cpu().numpy()[:, 0]
    assert np.array_equal(assoc, srv) and (srv >= 0).any()
    assert np.array_equal(qoe_ref.cents(util), k)
    tabs, _ = _cent_tabs(env.plan, 1, 0)
    lut = np.asarray(env.plan.classes[0]["rate_lut"], dtype=np.float64)
    bs = env.bs_xy.cpu().numpy().astype(np.int64)
    d2 = ((pts[:, None, :] - bs[None]) ** 2).sum(-1)
    want = np.where(srv >= 0, map_ref.shared_rate(lut, 1)[np.minimum(d2[np.arange(len(pts)), np.maximum(srv, 0)], len(lut) - 1)], 0.0)
    assert np.array_equal(rate, want)


@pytest.mark.gpu
def test_all_ues_on_one_point_agree_with_the_step_at_load_u():
    """FORK, generic kernel, MComCustom's per-env layouts: the 7 UEs of env e on grid point e share the map's
    serving BS at the load-7 rate and cent."""
    stride = 7
    env = _custom(29 * 29, generic_kernel=True)
    assert env.step_kernel_name == "step_kernel"
    U = env.plan.num_ues
    xs, ys = map_ref.grid(env.plan.width, env.plan.height, stride)
    X, Y = np.meshgrid(xs, ys)
    pts = np.stack([X.ravel(), Y.ravel()], axis=1)
    _placed(env, pts, U)
    m = env.layout_map(stride=stride, load=U)
    E = env.num_envs
    srv = m.serving.cpu().numpy().reshape(E, -1)[np.arange(E), np.arange(E)]
    k = m.qoe.cpu().numpy().reshape(E, -1)[np.arange(E), np.arange(E)]
    assoc, util = env.assoc.cpu().numpy(), env.utility_scaled.cpu().numpy()
    assert np.array_equal(assoc, np.repeat(srv[:, None], U, axis=1)) and (srv >= 0).sum() > E // 2
    assert np.array_equal(qoe_ref.cents(util), np.repeat(k[:, None], U, axis=1))
    bs = env.bs_xy.cpu().numpy().astype(np.int64)
    lut = map_ref.shared_rate(np.asarray(env.plan.classes[0]["rate_lut"], dtype=np.float64), U)
    d2 = ((pts - bs[np.arange(E), np.maximum(srv, 0)]) ** 2).sum(-1)
    want = np.where(srv >= 0, lut[np.minimum(d2, len(lut) - 1)], 0.0)
    assert np.array_equal(env.rate.cpu().numpy(), np.repeat(want[:, None], U, axis=1))


@pytest.mark.gpu
def test_layout_map_has_no_side_effects():
    import torch

    a, b = _custom(96), _custom(96)
    for s in range(3):
        a.step(0, s)
        b.step(0, s)
    bufs = lambda env: {**env.state_dict(), "metrics": env.metrics.clone()}  # noqa: E731
    before = bufs(a)
    for stride in (1, 4):
        a.layout_map(stride=stride, load=3, threshold=0.1)
        a.layout_map([0, 3, 200], stride=stride, maps=False)
    torch.cuda.synchronize()
    after = bufs(a)
    assert before.keys() == after.keys()
    for key in before:
        assert torch.equal(before[key], after[key]), key
    a.step(0, 3)
    b.step(0, 3)
    sa, sb = a.rollout(5, record=("pos", "assoc", "rate", "utility")), b.rollout(5, record=("pos", "assoc", "rate", "utility"))
    for key in sa:
        assert torch.equal(sa[key], sb[key]), key
    for key, v in bufs(a).items():
        assert torch.equal(v, bufs(b)[key]), key


@pytest.mark.gpu
def test_error_cases_return_a_message_and_write_nothing():
    import torch

    env = _custom(32)
    dev = env.device
    stats = torch.full((4, 6), 77, dtype=torch.int64, device=dev)
    area = torch.full((4 * env.plan.num_bs + 1,), 77, dtype=torch.int32, device=dev)
    maps = torch.full((3, 4, 200, 200), 77, dtype=torch.uint8, device=dev)
    ptr = lambda t, off=0: C.c_void_p(t.data_ptr() + off)  # noqa: E731

    def call(handle=env._handle, n=4, off_s=0, off_a=0, **kw):
        prm = _lib.MapParams(**{"stride": 1, "ue_class": 0, "load": 1, "threshold": 0.0, **kw})
        n0 = env.launch_count
        rc = env._lib.mbe_layout_map(handle, None, n, C.byref(prm), ptr(stats, off_s), ptr(area, off_a),
                                     ptr(maps[0]), ptr(maps[1]), ptr(maps[2]), env._stream())
        assert env.launch_count == n0
        return rc, env._lib.mbe_last_error().decode()

    unbound = object.__new__(type(env))
    unbound.plan, unbound.config, unbound.device, unbound._lib = env.plan, env.config, env.device, env._lib
    unbound._keepalive, unbound._handle = [], C.c_void_p()
    unbound._create_handle()
    cases = [
        (dict(handle=None), "null handle"),
        (dict(handle=unbound._handle), "mbe_bind has not been called"),
        (dict(n=-1), "n=-1"),
        (dict(stride=0), "stride=0"),
        (dict(load=0), "load=0"),
        (dict(ue_class=1), "ue_class=1"),
        (dict(ue_class=-1), "ue_class=-1"),
        (dict(threshold=float("nan")), "threshold must be finite"),
        (dict(threshold=float("inf")), "threshold must be finite"),
        (dict(off_s=4), "stats must be 8-byte aligned"),
        (dict(off_a=2), "area must be 4-byte aligned"),
    ]
    try:
        for kw, msg in cases:
            rc, err = call(**kw)
            assert rc != 0 and msg in err, (kw, err)
    finally:
        unbound.close()
    torch.cuda.synchronize()
    assert (stats == 77).all() and (area == 77).all() and (maps == 77).all()
    prm = _lib.MapParams(stride=1, ue_class=0, load=1, threshold=0.0)
    assert env._lib.mbe_layout_map(env._handle, None, 0, C.byref(prm), None, None, None, None, None, env._stream()) == 0


@pytest.mark.gpu
def test_map_result_of_a_four_trajectory_scorer_is_the_stats_of_rows_l_times_4():
    import torch
    from mobile_env_gan_b200.scoring import LayoutScorer

    env = _custom(256, num_trajectories=4)
    sc = LayoutScorer(env, low_qoe_threshold=0.1)
    L = sc.num_layouts
    xy, nbs = env.bs_xy.view(L, 4, -1, 2)[:, 0].clone(), env.nbs.view(L, 4)[:, 0].clone()
    env.bs_xy.view(L, 4, -1, 2).copy_(xy[:, None])
    env.nbs.view(L, 4).copy_(nbs[:, None])
    for load in (1, 7):
        got = sc.map_result(stride=2, load=load)
        full = env.layout_map(stride=2, load=load, threshold=0.1, maps=False)
        rows = full.stats.view(L, 4, 6)
        assert torch.equal(rows, rows[:, :1].expand(L, 4, 6))  # the replica rows hold the same layout
        want = full.result()
        for key, v in want.items():
            assert torch.equal(got[key], v[::4]), key
        assert torch.equal(got["Score"], torch.from_numpy(map_ref.result(full.stats[::4].cpu().numpy())["Score"]).to(v.device))
