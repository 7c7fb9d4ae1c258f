"""Layout evolution (mbe_evolve_layouts, DESIGN.md section 10): the properties of the operator on its
numpy restatement oracle/evolve_ref.py (CPU), the CUDA kernel against that restatement bit for bit,
the entry's argument checks, and the LayoutEvolution search on MComCustom (GPU)."""
import ctypes as C
import math

import numpy as np
import pytest

from oracle import evolve_ref as ER
from mobile_env_gan_b200 import _lib

OPS = dict(tournament_size=2, p_cross=0.5, p_move=0.3, step=7, p_add=0.2, p_del=0.2)


def random_population(rng, E, B, nmin, nmax, width, height):
    xm, ym = ER.coord_range(width, height)
    nbs = rng.integers(nmin, nmax + 1, size=E)
    xy = np.stack([rng.integers(0, xm + 1, size=(E, B)), rng.integers(0, ym + 1, size=(E, B))], axis=-1)
    xy[np.arange(B)[None, :] >= nbs[:, None]] = 0
    return xy.astype(np.int16), nbs.astype(np.int32)


def _evolve(xy, nbs, fit, elites=(), *, seed=7, generation=0, nmin=5, nmax=10, width=200.0, height=200.0,
            env_offset=0, **ops):
    kw = dict(OPS, **ops)
    return ER.evolve(xy, nbs, fit, np.asarray(elites, dtype=np.int64), seed=seed, generation=generation, nmin=nmin,
                     nmax=nmax, width=width, height=height, env_offset=env_offset, **kw)


# ------------------------------------------------------------------------------- CPU ----
@pytest.mark.parametrize("width,height", [(200.0, 200.0), (150.5, 99.25)])
def test_children_stay_on_the_map_with_counts_in_range_and_dead_slots_zero(width, height):
    rng = np.random.default_rng(1)
    E, B, nmin, nmax = 300, 12, 3, 12
    xy, nbs = random_population(rng, E, B, nmin, nmax, width, height)
    # parents on the map's edges make the clamps bite
    xm, ym = ER.coord_range(width, height)
    xy[::3, :, 0] = np.where(np.arange(B)[None, :] < nbs[::3, None], xm, 0)
    fit = rng.standard_normal(E).astype(np.float32)
    for g in range(3):
        cxy, cn = _evolve(xy, nbs, fit, generation=g, nmin=nmin, nmax=nmax, width=width, height=height,
                          step=40, p_move=0.7, p_add=0.4, p_del=0.4)
        assert ((cn >= nmin) & (cn <= nmax)).all()
        live = np.arange(B)[None, :] < cn[:, None]
        assert (cxy[..., 0][live] >= 0).all() and (cxy[..., 0][live] <= xm).all()
        assert (cxy[..., 1][live] >= 0).all() and (cxy[..., 1][live] <= ym).all()
        assert (cxy[~live] == 0).all()
        assert (cn != nbs).any()  # add / delete did fire
        xy, nbs = cxy, cn


def test_elites_are_verbatim_and_an_out_of_range_id_breeds():
    rng = np.random.default_rng(2)
    E, B = 64, 10
    xy, nbs = random_population(rng, E, B, 5, 10, 200, 200)
    fit = rng.standard_normal(E).astype(np.float32)
    elites = [5, 63, 0, E, -1]
    cxy, cn = _evolve(xy, nbs, fit, elites, p_move=1.0, step=30)
    for c, e in enumerate(elites[:3]):
        assert (cxy[c] == xy[e]).all() and cn[c] == nbs[e]
    bred, _ = _evolve(xy, nbs, fit, [], p_move=1.0, step=30)
    assert (cxy[3:] == bred[3:]).all()  # ids E and -1: ordinary children, the same draws as without elites


def test_no_operators_copy_a_uniformly_drawn_parent():
    rng = np.random.default_rng(3)
    E, B = 257, 10
    xy, nbs = random_population(rng, E, B, 5, 10, 200, 200)
    fit = rng.standard_normal(E).astype(np.float32)
    cxy, cn = _evolve(xy, nbs, fit, tournament_size=1, p_cross=0.0, p_move=0.0, p_add=0.0, p_del=0.0)
    G = np.arange(E, dtype=np.uint32)
    r0 = ER.philox4x32(G, 0, 0, ER.PURPOSE_EVOLVE, 7, 0)[0]
    parent = (r0.astype(np.uint64) * np.uint64(E)) >> np.uint64(32)
    assert (cxy == xy[parent]).all() and (cn == nbs[parent]).all()


def test_moves_with_step_zero_change_nothing():
    rng = np.random.default_rng(4)
    E, B = 128, 10
    xy, nbs = random_population(rng, E, B, 5, 10, 200, 200)
    fit = rng.standard_normal(E).astype(np.float32)
    a = _evolve(xy, nbs, fit, p_move=1.0, step=0)
    b = _evolve(xy, nbs, fit, p_move=0.0, step=0)
    assert (a[0] == b[0]).all() and (a[1] == b[1]).all()


def test_ties_go_to_the_smaller_index_and_nan_loses():
    fit = np.array([1.0, 3.0, np.nan, 3.0, -np.inf], dtype=np.float32)
    assert ER.tournament([1 << 30, 3 << 30, 0, 0], fit, 2) == 1  # candidates 1 and 3 tie at 3.0
    assert ER.tournament([3 << 30, 1 << 30, 0, 0], fit, 2) == 1
    assert ER.tournament([2 << 30, 0, 0, 0], fit, 2) == 0  # NaN (2) loses to 1.0 (0)
    nan = np.array([np.nan, -np.inf, np.nan, np.nan], dtype=np.float32)
    assert ER.tournament([3 << 30, 2 << 30, 1 << 30, 3 << 30], nan, 4) == 1  # all -inf: smallest index
    assert ER.tournament([3 << 30, 2 << 30, 0, 0], fit, 1) == 3  # T = 1: the first candidate


def test_same_generation_same_children_other_generation_different():
    rng = np.random.default_rng(5)
    E, B = 200, 10
    xy, nbs = random_population(rng, E, B, 5, 10, 200, 200)
    fit = rng.standard_normal(E).astype(np.float32)
    a, b, c = (_evolve(xy, nbs, fit, generation=g) for g in (3, 3, 4))
    assert (a[0] == b[0]).all() and (a[1] == b[1]).all()
    assert (a[0] != c[0]).any()
    d = _evolve(xy, nbs, fit, generation=3, seed=8)
    assert (a[0] != d[0]).any()


def test_evolve_params_struct_size_matches_the_library():
    lib = _lib.load()
    assert lib.mbe_struct_size(6) == C.sizeof(_lib.EvolveParams) == 56


# ------------------------------------------------------------------------------- GPU ----
def _custom(E, **cfg):
    from mobile_env_gan_b200.scenarios import MComCustom

    return MComCustom(config={"num_envs": E, **cfg})


def _params(seed, generation, T, p_cross, p_move, step, p_add, p_del):
    return _lib.EvolveParams(seed=seed, generation=generation, tournament=T, step=step, p_cross=p_cross,
                             p_move=p_move, p_add=p_add, p_del=p_del)


def _kernel(env, fit, xy, nbs, elites, prm):
    import torch

    dev = env.device
    t = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a)).to(device=dev, dtype=dt)  # noqa: E731
    fit_d, xy_d, nbs_d = t(fit, torch.float32), t(xy, torch.int16), t(nbs, torch.int32)
    el = t(np.asarray(elites, dtype=np.int32), torch.int32) if len(elites) else None
    cxy, cn = torch.full_like(xy_d, 0x7777), torch.full_like(nbs_d, -9)
    p = lambda x: None if x is None else C.c_void_p(x.data_ptr())  # noqa: E731
    before = env.launch_count
    _lib.check(env._lib.mbe_evolve_layouts(env._handle, p(fit_d), p(xy_d), p(nbs_d), p(el), len(elites),
                                           C.byref(prm), p(cxy), p(cn), env._stream()))
    assert env.launch_count == before + 1
    return cxy.cpu().numpy(), cn.cpu().numpy()


CASES = [  # E, config, T, K, (p_cross, p_move, step, p_add, p_del), fitness kind
    (1, {}, 1, 0, (0.5, 0.5, 5, 0.5, 0.5), "normal"),
    (1, {}, 2, 1, (1.0, 1.0, 9, 1.0, 1.0), "normal"),
    (100, {}, 1, 0, (0.0, 0.0, 0, 0.0, 0.0), "normal"),
    (100, {}, 2, 1, (1.0, 1.0, 12, 1.0, 0.0), "ties"),
    (333, {"env_offset": 4096}, 3, 333, (0.4, 0.3, 7, 0.2, 0.3), "nan"),
    (333, {"env_offset": 4096}, 3, 17, (0.4, 0.3, 7, 0.0, 1.0), "nan"),
    (1 << 16, {}, 4, 1024, (0.5, 0.2, 10, 0.1, 0.1), "ties"),
    (1000, {"bs_random": (3, 40), "max_bs": 40}, 4, 5, (0.6, 0.5, 30, 0.3, 0.3), "normal"),
    (1000, {"bs_random": (3, 40), "max_bs": 40}, 2, 0, (1.0, 1.0, 32767, 1.0, 1.0), "nan"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("E,cfg,T,K,ops,kind", CASES)
def test_kernel_equals_restatement_bit_for_bit(E, cfg, T, K, ops, kind):
    env = _custom(E, **cfg)
    p = env.plan
    B, (nmin, nmax) = p.num_bs, p.bs_random
    rng = np.random.default_rng(E + T + K)
    xy, nbs = random_population(rng, E, B, nmin, nmax, p.width, p.height)
    if kind == "ties":
        fit = rng.integers(0, 4, size=E).astype(np.float32)
    else:
        fit = rng.standard_normal(E).astype(np.float32)
        if kind == "nan":
            fit[rng.random(E) < 0.3] = np.nan
    elites = rng.permutation(E)[:K].astype(np.int64)
    if K > 2:
        elites[1], elites[2] = E + 3, -1  # out-of-range ids: ordinary children
    p_cross, p_move, step, p_add, p_del = ops
    for gen in (0, 5):
        got = _kernel(env, fit, xy, nbs, elites, _params(11, gen, T, p_cross, p_move, step, p_add, p_del))
        want = ER.evolve(xy, nbs, fit, elites, seed=11, generation=gen, tournament_size=T, p_cross=p_cross,
                         p_move=p_move, step=step, p_add=p_add, p_del=p_del, nmin=nmin, nmax=nmax, width=p.width,
                         height=p.height, env_offset=p.env_offset)
        assert np.array_equal(got[1], want[1])
        assert np.array_equal(got[0], want[0])


@pytest.mark.gpu
def test_kernel_equals_restatement_on_a_non_integer_map():
    env = _custom(500, width=150.5, height=99.25, movement_params={"width": 150.5, "height": 99.25,
                                                                    "reset_rng_episode": True})
    p = env.plan
    assert (p.width, p.height) == (150.5, 99.25)
    rng = np.random.default_rng(9)
    xy, nbs = random_population(rng, 500, p.num_bs, *p.bs_random, p.width, p.height)
    xy[::2, :, 0] = np.where(np.arange(p.num_bs)[None, :] < nbs[::2, None], 150, 0)
    fit = rng.standard_normal(500).astype(np.float32)
    got = _kernel(env, fit, xy, nbs, [], _params(3, 1, 2, 0.5, 0.8, 20, 0.6, 0.2))
    want = ER.evolve(xy, nbs, fit, [], seed=3, generation=1, tournament_size=2, p_cross=0.5, p_move=0.8, step=20,
                     p_add=0.6, p_del=0.2, nmin=p.bs_random[0], nmax=p.bs_random[1], width=p.width, height=p.height)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])


@pytest.mark.gpu
def test_entry_rejects_bad_arguments_and_leaves_parents_untouched():
    import torch

    env = _custom(256)
    E, B = 256, env.plan.num_bs
    rng = np.random.default_rng(0)
    xy_h, nbs_h = random_population(rng, E, B, 5, 10, 200, 200)
    xy, nbs = torch.from_numpy(xy_h).cuda(), torch.from_numpy(nbs_h).cuda()
    fit = torch.randn(E, device="cuda")
    el = torch.arange(4, dtype=torch.int32, device="cuda")
    cxy, cn = torch.zeros_like(xy), torch.zeros_like(nbs)
    big = torch.zeros(2 * E * B * 2 + 8, dtype=torch.int16, device="cuda")
    p = lambda x: None if x is None else C.c_void_p(x.data_ptr())  # noqa: E731
    ok = dict(T=2, p_cross=0.5, p_move=0.5, step=5, p_add=0.1, p_del=0.1)

    def call(env=env, fit=fit, xy=xy, nbs=nbs, el=el, k=4, cxy=cxy, cn=cn, raw_cxy=None, **over):
        kw = dict(ok, **over)
        prm = _params(1, 0, kw["T"], kw["p_cross"], kw["p_move"], kw["step"], kw["p_add"], kw["p_del"])
        cx = raw_cxy if raw_cxy is not None else p(cxy)
        rc = env._lib.mbe_evolve_layouts(env._handle, p(fit), p(xy), p(nbs), p(el), k, C.byref(prm), cx, p(cn),
                                         env._stream())
        return rc, env._lib.mbe_last_error().decode()

    assert call()[0] == 0
    bad = [
        (dict(fit=None), "null"), (dict(xy=None), "null"), (dict(cn=None), "null"),
        (dict(k=-1), "n_elite"), (dict(k=E + 1), "n_elite"), (dict(el=None), "elite_ids"),
        (dict(T=0), "tournament"), (dict(T=5), "tournament"), (dict(step=-1), "step"), (dict(step=32768), "step"),
        (dict(p_cross=-0.1), "probability"), (dict(p_move=1.5), "probability"), (dict(p_add=math.nan), "probability"),
        (dict(p_del=math.inf), "probability"),
        (dict(cxy=xy), "overlap"), (dict(cn=nbs), "overlap"), (dict(cn=fit.view(torch.int32)), "overlap"),
        (dict(raw_cxy=C.c_void_p(xy.data_ptr() + 4 * (E * B - 1))), "overlap"),
        (dict(raw_cxy=C.c_void_p(big.data_ptr() + 2)), "aligned"),
    ]
    for over, word in bad:
        rc, msg = call(**over)
        assert rc != 0 and word in msg, (over, msg)
    from mobile_env_gan_b200.scenarios import MComSmall

    shared = MComSmall(config={"num_envs": 64, "mode": "fork"})
    rc, msg = call(env=shared)
    assert rc != 0 and "per-env" in msg
    torch.cuda.synchronize()
    assert np.array_equal(xy.cpu().numpy(), xy_h) and np.array_equal(nbs.cpu().numpy(), nbs_h)


def _fresh_score(xy, nbs):
    """Scores layouts on a fresh MComCustom batch (one env per layout)."""
    from mobile_env_gan_b200.scoring import LayoutScorer

    env = _custom(xy.shape[0])
    env.reset()
    env.set_station_positions(xy, nbs)
    sc = LayoutScorer(env)
    sc.run_episode()
    return env, sc.result()["Score"]


@pytest.mark.gpu
def test_layout_evolution_on_custom():
    import torch
    from mirror import Mirror
    from mobile_env_gan_b200.scoring import LayoutEvolution

    E, G = 4096, 10
    env = _custom(E)
    evo = LayoutEvolution(env, seed=5)
    K = evo.elites
    prev_fit, prev_elites, bests = None, None, []
    for g in range(G):
        fit = evo.step().clone()
        if prev_fit is not None:  # the elites come first and keep their scores bit for bit
            assert torch.equal(fit[:K], prev_fit[prev_elites.long()])
        bests.append(float(fit.max()))
        prev_fit, prev_elites = fit, evo.elite_ids.clone()
    assert all(b2 >= b1 for b1, b2 in zip(bests, bests[1:]))
    # generation 0 is plain random search over E layouts; evolution is expected to beat it
    assert bests[-1] > bests[0], bests

    other = LayoutEvolution(_custom(E), seed=5)
    assert other.run(G) == bests
    for a, b in zip(evo.population(), other.population()):
        assert torch.equal(a, b)

    # the winners replayed through the oracle mirror reproduce their scores
    xy, nbs, score = evo.best(8)
    assert torch.equal(score, torch.sort(score, descending=True).values)
    env8 = _custom(8)
    mir = Mirror(env8)
    env8.reset(), mir.reset()
    mir.bs, mir.nbs = xy.cpu().numpy().astype(np.int64), nbs.cpu().numpy().astype(np.int64)
    qoe = [np.round(mir.step_fork()["utility"], 2) for _ in range(env8.plan.ep_time)]
    q = np.concatenate(qoe, axis=1)
    want = q.mean(axis=1) - 0.1 * q.var(axis=1) - 10.0 * (q < 0.0).mean(axis=1)
    np.testing.assert_allclose(score.cpu().numpy(), want, atol=1e-5, rtol=0)
    assert np.abs(score.cpu().numpy() - want).mean() < 2e-3
    _, fresh = _fresh_score(xy.repeat(4, 1, 1), nbs.repeat(4))  # 32 envs: the same fused kernel
    assert torch.equal(fresh.view(4, 8), score.expand(4, 8))


@pytest.mark.gpu
def test_env_still_steps_rolls_out_and_renders_after_a_search():
    import torch
    from mobile_env_gan_b200.scoring import LayoutEvolution

    E = 256
    env = _custom(E)
    evo = LayoutEvolution(env, seed=1, elites=4)
    evo.run(3)
    xy, nbs = (t.clone() for t in evo.population())
    ref = _custom(E)
    for e in (env, ref):
        e.reset()
        e.set_station_positions(xy, nbs)
    for k in range(3):
        env.step(0, k), ref.step(0, k)
        assert torch.equal(env.assoc, ref.assoc) and torch.equal(env.rate, ref.rate)
    sa, sb = env.rollout(5, record=("pos", "assoc")), ref.rollout(5, record=("pos", "assoc"))
    assert torch.equal(sa["assoc"], sb["assoc"]) and torch.equal(sa["pos"], sb["pos"])
    ids = torch.arange(0, E, 37, dtype=torch.int32, device=env.device)
    assert torch.equal(env.render_frames(ids, (64, 64)), ref.render_frames(ids, (64, 64)))


@pytest.mark.gpu
def test_layout_evolution_rejects_unsuitable_envs_and_populations():
    from mobile_env_gan_b200.scenarios import MComSmall
    from mobile_env_gan_b200.scoring import LayoutEvolution

    with pytest.raises(ValueError, match="per-env"):
        LayoutEvolution(MComSmall(config={"num_envs": 32, "mode": "fork"}))
    with pytest.raises(ValueError, match="FORK"):
        LayoutEvolution(_custom(32, mode="gym"))
    with pytest.raises(ValueError, match="trajectory"):
        LayoutEvolution(_custom(32, shared_trajectory=False))
    env = _custom(32)
    rng = np.random.default_rng(0)
    xy, nbs = random_population(rng, 32, 10, 5, 10, 200, 200)
    LayoutEvolution(env, bs_xy=xy, nbs=nbs)
    with pytest.raises(ValueError, match="nbs"):
        LayoutEvolution(env, bs_xy=xy, nbs=np.full(32, 11))
    bad = xy.copy()
    bad[0, 0] = (200, 0)
    with pytest.raises(ValueError, match="coordinates"):
        LayoutEvolution(env, bs_xy=bad, nbs=nbs)
    with pytest.raises(ValueError, match="population"):
        LayoutEvolution(env, bs_xy=xy[:5], nbs=nbs[:5])
