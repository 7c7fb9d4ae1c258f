"""Layouts scored over M UE trajectories (``num_trajectories``, DESIGN.md section 10): the host plan's
rules (CPU); on the GPU the env-to-trajectory mapping g mod M bit for bit, M = 1 as today, the pooled
score against the oracle mirror, placement independence of a layout's score, the entry points' checks,
mbe_evolve_layouts over the L = num_envs / M layouts against oracle/evolve_ref.py, and LayoutEvolution /
LayoutScorer.score_layouts with M = 4."""
import ctypes as C
import dataclasses

import numpy as np
import pytest

from oracle import evolve_ref as ER
from mobile_env_gan_b200 import _lib
from mobile_env_gan_b200.core.base import MComCore, Plan
from mobile_env_gan_b200.core.entities import UserEquipment
from mobile_env_gan_b200.core.util import deep_dict_merge
from mobile_env_gan_b200.scenarios.custom import MComCustom


def plan_of(extra):
    cfg = MComCustom.seeding(deep_dict_merge(MComCustom.default_config(), extra))
    users = [UserEquipment(i, **cfg["ue"]) for i in range(MComCustom.NUM_UES)]
    return MComCustom.build_plan([], users, cfg)


def _same(a, b):
    if isinstance(a, np.ndarray) or isinstance(b, np.ndarray):
        return np.array_equal(a, b)
    if isinstance(a, dict):
        return a.keys() == b.keys() and all(_same(a[k], b[k]) for k in a)
    if isinstance(a, (list, tuple)):
        return len(a) == len(b) and all(_same(x, y) for x, y in zip(a, b))
    return a == b


def random_population(rng, L, B, nmin, nmax, width, height):
    xm, ym = ER.coord_range(width, height)
    nbs = rng.integers(nmin, nmax + 1, size=L)
    xy = np.stack([rng.integers(0, xm + 1, size=(L, B)), rng.integers(0, ym + 1, size=(L, B))], axis=-1)
    xy[np.arange(B)[None, :] >= nbs[:, None]] = 0
    return xy.astype(np.int16), nbs.astype(np.int32)


# ------------------------------------------------------------------------------- CPU ----
@pytest.mark.parametrize("M", [1, 2, 8, 32])
def test_plan_accepts_power_of_two_trajectory_counts(M):
    p = plan_of({"num_envs": 64, "num_trajectories": M, "env_offset": 3 * 32})
    assert p.num_trajectories == M and p.shared_trajectory


@pytest.mark.parametrize("extra,word", [
    ({"num_envs": 63, "num_trajectories": 3}, "power of two"),
    ({"num_envs": 64, "num_trajectories": 8, "shared_trajectory": False}, "shared_trajectory"),
    ({"num_envs": 64, "num_trajectories": 8, "movement_params": {"reset_rng_episode": False}}, "shared_trajectory"),
    ({"num_envs": 36, "num_trajectories": 8}, "multiple"),
    ({"num_envs": 4, "num_trajectories": 8}, "multiple"),
    ({"num_envs": 64, "num_trajectories": 8, "env_offset": 4}, "env_offset"),
    ({"num_envs": 64, "num_trajectories": 0}, ">= 1"),
])
def test_plan_rejects_each_broken_rule(extra, word):
    with pytest.raises(ValueError, match=word):
        plan_of(extra)


def test_default_plan_is_todays():
    assert Plan.__dataclass_fields__["num_trajectories"].default == 1
    assert MComCore.default_config()["num_trajectories"] == 1
    a, b = plan_of({"num_envs": 64}), plan_of({"num_envs": 64, "num_trajectories": 1})
    for f in dataclasses.fields(Plan):
        assert _same(getattr(a, f.name), getattr(b, f.name)), f.name
    assert a.num_trajectories == 1


def test_config_struct_size_matches_the_library():
    lib = _lib.load()
    assert lib.mbe_struct_size(0) == C.sizeof(_lib.Config)
    assert _lib.Config.num_trajectories.offset == _lib.Config.num_ue_classes.offset + 4


# ------------------------------------------------------------------------------- GPU ----
def _custom(E, **cfg):
    return MComCustom(config={"num_envs": E, **cfg})


def _bytes(t):
    import torch

    return t.contiguous().view(-1).view(torch.uint8)


@pytest.mark.gpu
@pytest.mark.parametrize("M,offset", [(8, 0), (8, 8 * 513), (2, 2 * 77)])
def test_custom_env_e_follows_independent_trajectory_e_mod_m(M, offset):
    import torch

    E, T = 256, 20
    env = _custom(E, num_trajectories=M, env_offset=offset)
    ref = _custom(M, shared_trajectory=False)
    assert not ref.plan.shared_trajectory
    env.reset(), ref.reset()
    U = env.NUM_USERS
    assert torch.equal(env.pos.view(E // M, M, U, 2), ref.pos[None].expand(E // M, M, U, 2))
    got, want = env.rollout(T, record=("pos", "wp")), ref.rollout(T, record=("pos", "wp"))
    for k in ("pos", "wp"):
        assert torch.equal(got[k].view(T, E // M, M, U, 2), want[k][:, None].expand(T, E // M, M, U, 2)), k
    # the same through env windows: the mask applies to the global id of every window
    env.reset(), ref.reset()
    for _ in range(T):
        env.step_window(0, 64)
        env.step_window(64, E - 64)
        ref.step(0, 0)
        assert torch.equal(env.pos.view(E // M, M, U, 2), ref.pos[None].expand(E // M, M, U, 2))
        assert torch.equal(env.wp.view(E // M, M, U, 2), ref.wp[None].expand(E // M, M, U, 2))


@pytest.mark.gpu
def test_gym_env_e_follows_independent_trajectory_e_mod_m():
    import torch

    import mobile_env_gan_b200 as mbe

    M, E = 4, 64
    env = mbe.make("mobile-medium-central-v0", num_envs=E, env_offset=4 * M,
                   config={"shared_trajectory": True, "num_trajectories": M})
    ref = mbe.make("mobile-medium-central-v0", num_envs=M)
    assert env.plan.mode == _lib.MODE_GYM and not ref.plan.shared_trajectory
    env.reset(), ref.reset()
    U = env.NUM_USERS
    for _ in range(20):
        env.step(torch.zeros(E, U, dtype=torch.int32, device=env.device))
        ref.step(torch.zeros(M, U, dtype=torch.int32, device=ref.device))
        assert torch.equal(env.pos.view(E // M, M, U, 2), ref.pos[None].expand(E // M, M, U, 2))
        assert torch.equal(env.wp.view(E // M, M, U, 2), ref.wp[None].expand(E // M, M, U, 2))


@pytest.mark.gpu
def test_one_trajectory_is_todays_env_byte_for_byte():
    import torch

    E = 512
    a, b = _custom(E, env_offset=96), _custom(E, env_offset=96, num_trajectories=1)
    acc = [torch.zeros(E, 4, device="cuda") for _ in range(2)]
    names = ("pos", "wp", "assoc", "rate", "utility")
    for env in (a, b):
        env.reset()
    for k, v in a.state_dict().items():
        assert torch.equal(_bytes(v), _bytes(b.state_dict()[k])), k
    sa, sb = a.rollout(20, qoe_acc=acc[0], record=names), b.rollout(20, qoe_acc=acc[1], record=names)
    for k in names:
        assert torch.equal(_bytes(sa[k]), _bytes(sb[k])), k
    assert torch.equal(_bytes(acc[0]), _bytes(acc[1]))
    for k, v in a.state_dict().items():
        assert torch.equal(_bytes(v), _bytes(b.state_dict()[k])), k


def _replicate(env, M):
    """Copies layout row l*M to the other M - 1 replica rows of layout l; returns (bs_xy [L,B,2], nbs [L])."""
    L, B = env.num_envs // M, env.plan.num_bs
    xy, n = env.bs_xy.view(L, M, B, 2)[:, 0].clone(), env.nbs.view(L, M)[:, 0].clone()
    env.bs_xy.view(L, M, B, 2).copy_(xy[:, None])
    env.nbs.view(L, M).copy_(n[:, None])
    return xy, n


@pytest.mark.gpu
def test_assoc_rates_and_pooled_scores_match_the_mirror():
    from mirror import Mirror
    from mobile_env_gan_b200.scoring import LayoutScorer

    M, E = 4, 256
    L = E // M
    env = _custom(E, num_trajectories=M, env_offset=M * 40)
    mir = Mirror(env)
    mir.traj_gid = mir.gid & (M - 1)
    env.reset(), mir.reset()
    assert np.array_equal(env.pos.cpu().numpy(), mir.pos)
    xy, nbs = _replicate(env, M)
    mir.bs, mir.nbs = env.bs_xy.cpu().numpy().astype(np.int64), env.nbs.cpu().numpy().astype(np.int64)
    sc = LayoutScorer(env)
    assert sc.num_layouts == L
    qoe = []
    for k in range(env.plan.ep_time):
        env.step(0, k)
        sc.update()
        out = mir.step_fork()
        assert np.array_equal(env.assoc.cpu().numpy(), out["assoc"]), k
        assert np.array_equal(env.rate.cpu().numpy(), out["rate"]), k
        assert np.array_equal(env.pos.cpu().numpy(), out["pos_after"]), k
        qoe.append(np.round(out["utility"], 2))
    q = np.concatenate(qoe, axis=1).reshape(L, -1)  # rows l*M .. l*M + M-1 of layout l, side by side
    want = q.mean(axis=1) - 0.1 * q.var(axis=1) - 10.0 * (q < 0.0).mean(axis=1)
    for score in (sc.result()["Score"], LayoutScorer(env).score_layouts(xy, nbs)):
        assert score.shape == (L,)
        np.testing.assert_allclose(score.cpu().numpy(), want, atol=1e-5, rtol=0)
        assert np.abs(score.cpu().numpy() - want).mean() < 2e-3
    idx, top = sc.best(5)
    assert int(idx.max()) < L


@pytest.mark.gpu
def test_a_layouts_pooled_score_does_not_depend_on_where_it_runs():
    import torch
    from mobile_env_gan_b200.scoring import LayoutScorer

    M = 4
    rng = np.random.default_rng(7)
    a = _custom(64 * M, num_trajectories=M)
    b = _custom(32 * M, num_trajectories=M, env_offset=M * 1000)
    xa, na = random_population(rng, 64, 10, 5, 10, 200, 200)
    xb, nb = random_population(rng, 32, 10, 5, 10, 200, 200)
    for i in (3, 50):
        xa[i], na[i] = xa[0], na[0]
    xb[7], nb[7] = xa[0], na[0]
    sa = LayoutScorer(a).score_layouts(xa, na)
    sb = LayoutScorer(b).score_layouts(xb, nb)
    assert torch.equal(_bytes(sa[[0, 3, 50]]), _bytes(sa[0].repeat(3)))
    assert torch.equal(_bytes(sb[7]), _bytes(sa[0]))
    assert len(set(sa.cpu().tolist())) > 32  # the other layouts score differently


def _create_fails(env, **plan):
    """mbe_create on env's plan with fields replaced; returns the error message."""
    keep = env._handle
    env.plan, old = dataclasses.replace(env.plan, **plan), env.plan
    env._handle = C.c_void_p()
    try:
        with pytest.raises(_lib.MbeError) as err:
            env._create_handle()
    finally:
        env.plan, env._handle = old, keep
    return str(err.value)


@pytest.mark.gpu
def test_create_rejects_bad_trajectory_counts_and_offsets():
    env = _custom(64, num_trajectories=8)
    bad = [
        (dict(num_trajectories=3), "power of two"),
        (dict(num_trajectories=-1), ">= 0"),
        (dict(shared_trajectory=False), "SHARED_TRAJECTORY"),
        (dict(num_trajectories=128), "exceeds num_envs"),
        (dict(num_envs=36), "multiple of num_trajectories"),
        (dict(env_offset=4), "env_offset"),
    ]
    for over, word in bad:
        msg = _create_fails(env, **over)
        assert word in msg, (over, msg)
    env.reset()
    env.rollout(2)  # the handle it kept still runs


def _evolve_call(env, fit, xy, nbs, elites, prm):
    import torch

    dev = env.device
    t = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a)).to(device=dev, dtype=dt)  # noqa: E731
    fit_d, xy_d, nbs_d = t(fit, torch.float32), t(xy, torch.int16), t(nbs, torch.int32)
    el = t(np.asarray(elites, dtype=np.int32), torch.int32)
    cxy, cn = torch.full_like(xy_d, 0x7777), torch.full_like(nbs_d, -9)
    p = lambda x: C.c_void_p(x.data_ptr())  # noqa: E731
    rc = env._lib.mbe_evolve_layouts(env._handle, p(fit_d), p(xy_d), p(nbs_d), p(el), len(elites), C.byref(prm),
                                     p(cxy), p(cn), env._stream())
    return rc, env._lib.mbe_last_error().decode(), cxy.cpu().numpy(), cn.cpu().numpy()


@pytest.mark.gpu
def test_evolve_breeds_layouts_with_offset_env_offset_over_m():
    M, L = 4, 333
    env = _custom(L * M, num_trajectories=M, env_offset=M * 1024)
    p = env.plan
    B, (nmin, nmax) = p.num_bs, p.bs_random
    rng = np.random.default_rng(11)
    xy, nbs = random_population(rng, L, B, nmin, nmax, p.width, p.height)
    fit = rng.standard_normal(L).astype(np.float32)
    fit[rng.random(L) < 0.2] = np.nan
    prm = _lib.EvolveParams(seed=9, generation=3, tournament=3, step=7, p_cross=0.4, p_move=0.3, p_add=0.2,
                            p_del=0.3)
    for K in (0, 17, L):
        elites = rng.permutation(L)[:K]
        rc, msg, cxy, cn = _evolve_call(env, fit, xy, nbs, elites, prm)
        assert rc == 0, msg
        want = ER.evolve(xy, nbs, fit, elites.astype(np.int64), seed=9, generation=3, tournament_size=3, p_cross=0.4,
                         p_move=0.3, step=7, p_add=0.2, p_del=0.3, nmin=nmin, nmax=nmax, width=p.width,
                         height=p.height, env_offset=p.env_offset // M)
        assert np.array_equal(cn, want[1]) and np.array_equal(cxy, want[0]), K
    rc, msg, _, _ = _evolve_call(env, fit, xy, nbs, np.arange(L + 1) % L, prm)
    assert rc != 0 and "n_elite" in msg and str(L) in msg


@pytest.mark.gpu
def test_layout_evolution_over_four_trajectories():
    import torch
    from mobile_env_gan_b200.scoring import LayoutEvolution, LayoutScorer

    M, L, G = 4, 1024, 8
    env = _custom(L * M, num_trajectories=M)
    evo = LayoutEvolution(env, seed=5)
    K = evo.elites
    assert K == L // 64 and evo.population()[0].shape == (L, env.plan.num_bs, 2)
    prev_fit, prev_elites, bests = None, None, []
    for g in range(G):
        fit = evo.step().clone()
        assert fit.shape == (L,)
        if prev_fit is not None:  # elites come first and keep their pooled scores bit for bit
            assert torch.equal(fit[:K], prev_fit[prev_elites.long()])
        bests.append(float(fit.max()))
        prev_fit, prev_elites = fit, evo.elite_ids.clone()
    assert all(b2 >= b1 for b1, b2 in zip(bests, bests[1:]))
    assert bests[-1] > bests[0], bests

    other = LayoutEvolution(_custom(L * M, num_trajectories=M), seed=5)
    assert other.run(G) == bests
    for a, b in zip(evo.population(), other.population()):
        assert torch.equal(a, b)

    xy, nbs, score = evo.best(8)
    fresh = LayoutScorer(_custom(8 * M, num_trajectories=M)).score_layouts(xy, nbs)
    assert torch.equal(fresh, score)

    # held out: 16 trajectories of another movement seed
    held_env = _custom(8 * 16, num_trajectories=16, seed=99)
    held = LayoutScorer(held_env)
    h1 = held.score_layouts(xy, nbs).clone()
    h2 = held.score_layouts(xy.cpu().numpy(), nbs.cpu().numpy())
    assert torch.equal(h1, h2)
    train_env = _custom(8 * 16, num_trajectories=16)
    train_env.reset(), held_env.reset()
    assert not torch.equal(train_env.pos[:16], held_env.pos[:16])
    assert not torch.equal(h1, LayoutScorer(train_env).score_layouts(xy, nbs))
    with pytest.raises(ValueError, match="population"):
        held.score_layouts(xy[:5], nbs[:5])
