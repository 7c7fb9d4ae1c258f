"""The QoE statistics behind the layout score (chooseBaseStation.ipynb ``qoeValue``) against the FP64
restatement ``oracle/qoe_ref.py``: the cent of every value, the low-QoE count at cent thresholds and the
sums, for ``qoe_accumulate_kernel`` (``LayoutScorer.update``) and the fused episode (``mbe_rollout``).

The contract (include/mbe.h ``mbe_accumulate_qoe``): the cent k is the exact half-even rounding of the FP32
utility times 100, the value is float32(k / 100) and it is low when float32(k / 100) < float32(threshold).
Counts must be exact; the FP32 sums must lie within a bound derived from their summation order."""
from __future__ import annotations

from fractions import Fraction

import numpy as np
import pytest

from oracle import qoe_ref as R

DEFAULT_UTILITY = (-20, 20, (10, 0, 10))  # every shipped scenario
EPISODE_THRESHOLDS = (0.0, 0.1, 0.3, -0.05, 0.5)


# ------------------------------------------------------------------------------------------- CPU --
def test_restatement_is_pythons_two_decimal_round_and_threshold_test():
    u = R.near_cents_and_ties(64)
    py = np.array([round(float(x), 2) for x in u])
    k = R.cents(u)
    assert np.array_equal(k / 100, py)
    assert np.array_equal(np.abs(k), np.rint(np.abs(k)))
    for c in range(-100, 101):
        t = c / 100
        assert np.array_equal(R.is_low(k, t), py < t), t
        # a threshold that rounds to the same float32 as a cent acts as that cent
        assert np.array_equal(R.is_low(k, float(np.float32(t))), py < t), t
    # the FP32 shortcut k * 0.01f is not float32(k / 100) for 60 cents, e.g. 10 * 0.01f < 0.1f
    wrong = [c for c in range(-100, 101) if np.float32(np.float32(c) * np.float32(0.01)) != R.cent_value(c)]
    assert len(wrong) == 60 and 10 in wrong and 30 in wrong
    # and rintf(u * 100.0f) rounds the FP32 product: off by a cent on 56 values in (0, 1] and their negatives
    old = np.rint((u * np.float32(100)).astype(np.float32))
    assert int(np.sum(old != k)) == 112 and R.cents(np.float32(0.015)) == 1


def _fmaf(a, b, c):
    """FP32 fused multiply-add; exact here because every product and sum below fits an FP64 mantissa."""
    return np.float32(Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c)))


def test_fp32_cent_helper_arithmetic_equals_the_restatement():
    """The steps of ``qoe_cent_value`` (mbe_device.cuh) in exact arithmetic, on every value near a cent
    or a half-cent tie: the cent and the corrected quotient float32(k / 100)."""
    f32 = np.float32
    u = R.near_cents_and_ties(8)
    p = (u * f32(100)).astype(f32)
    k = np.rint(p)
    for i in np.flatnonzero(np.abs(p - k) == f32(0.5)):
        e = _fmaf(u[i], f32(100), -p[i])
        if e != 0:
            k[i] = p[i] + np.copysign(f32(0.5), e)
    assert np.array_equal(k.astype(np.float64), R.cents(u))
    for c in range(-100, 101):
        q0 = f32(f32(c) * f32(0.01))
        r = _fmaf(-q0, f32(100), f32(c))
        exact = Fraction(float(r)) * Fraction(float(f32(0.01))) + Fraction(float(q0))
        q = f32(exact)
        if Fraction(float(q)) != exact:  # f32(Fraction) goes through FP64: check the rounding is to nearest
            lo, hi = np.nextafter(q, f32(-2)), np.nextafter(q, f32(2))
            assert abs(exact - Fraction(float(q))) < min(abs(exact - Fraction(float(lo))), abs(exact - Fraction(float(hi))))
        assert q == R.cent_value(c), c


def test_qoe_value_is_the_notebook_formula():
    rng = np.random.default_rng(3)
    u = rng.uniform(-1, 1, size=(50, 140)).astype(np.float32)
    q = np.vectorize(lambda x: round(float(x), 2))(u)
    for t in (0.0, 0.1, -0.05):
        got = R.qoe_value(*R.accumulate(u, t))
        np.testing.assert_allclose(got["Average QoE"], q.mean(axis=1), rtol=0, atol=1e-13)
        np.testing.assert_allclose(got["QoE Variance"], q.var(axis=1), rtol=0, atol=1e-13)
        assert np.array_equal(got["Low QoE Proportion"], (q < t).mean(axis=1))
        want = q.mean(axis=1) - 0.1 * q.var(axis=1) - 10.0 * (q < t).mean(axis=1)
        np.testing.assert_allclose(got["Score"], want, rtol=0, atol=1e-12)


def test_tie_margin_of_the_default_utility_exceeds_the_device_error_bound():
    """The kernels' FP32 utility (``scaled_utility``: SFU lg2.approx within 2^-22 * max(1, |log2 x|), plus
    FP32 roundings) must stay closer to the FP64 utility than the nearest half-cent tie, or a kernel cent can
    differ from the cent of the dump files.  Rates above 100 saturate the default utility at exactly 1."""
    margin = R.tie_margin(DEFAULT_UTILITY, 100.0)
    bound = R.device_utility_error_bound(DEFAULT_UTILITY, 100.0)
    assert 1e-6 < margin < 2e-6  # closest: rate 61.66
    assert margin == R.tie_margin(DEFAULT_UTILITY, 2e9)
    assert 0 < bound < margin / 2 and R.device_utility_error_bound(DEFAULT_UTILITY, 2e9) < margin / 2
    assert R.saturation_rate(DEFAULT_UTILITY, 2e9) == 100.01


# ------------------------------------------------------------------------------------------- GPU --
def _sum_bounds(u, depth):
    """Allowed |s1 - exact| and |s2 - exact| per row of QoE values u [rows, n] (FP32 values)."""
    q = R.cents(u) / 100
    return (R.sum_error_bound(np.abs(q).sum(axis=-1), depth),
            R.sum_error_bound((q * q).sum(axis=-1), depth, rel_term=3 * R.F32_EPS))


def _check_acc(acc, u, threshold, depth, what):
    """acc [rows, 4] from the device against the restatement of the values u [rows, n] behind it."""
    s1, s2, low, n = R.accumulate(u, threshold)
    e1, e2 = _sum_bounds(u, depth)
    acc = acc.astype(np.float64)
    assert np.array_equal(acc[:, 3], n), what
    bad = np.flatnonzero(acc[:, 2] != low)
    assert bad.size == 0, f"{what}: low count of {bad.size} rows, e.g. row {bad[:1]}: {acc[bad[:1], 2]} != {low[bad[:1]]}"
    assert np.all(np.abs(acc[:, 0] - s1) <= e1), (what, np.max(np.abs(acc[:, 0] - s1) - e1))
    assert np.all(np.abs(acc[:, 1] - s2) <= e2), (what, np.max(np.abs(acc[:, 1] - s2) - e2))
    return (s1, s2, low, n), (e1, e2)


def _core_env(U, E):
    from mobile_env_gan_b200.core.base import MComCore
    from mobile_env_gan_b200.core.entities import BaseStation, UserEquipment

    cfg = MComCore.default_config()
    stations = [BaseStation(i, xy, **cfg["bs"]) for i, xy in enumerate([(50, 50), (150, 50), (50, 150), (150, 150)])]
    users = [UserEquipment(i, **cfg["ue"]) for i in range(U)]
    return MComCore(stations, users, {"num_envs": E, "mode": "fork"})


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["custom-64", "70-ues", "custom-37"])
def test_accumulate_kernel_on_values_at_cents_and_ties(shape):
    """Values within 4 ulps of every cent and half-cent tie (and +-0, +-1) written into the utility
    buffer, at every cent threshold: MComCustom, a shape with U > 32 (the lane-strided loop) and an env
    count that is not a multiple of the 4 warps of a block."""
    import torch
    from mobile_env_gan_b200.scenarios import MComCustom
    from mobile_env_gan_b200.scoring import LayoutScorer

    env = {"custom-64": lambda: MComCustom(config={"num_envs": 64}), "70-ues": lambda: _core_env(70, 42),
           "custom-37": lambda: MComCustom(config={"num_envs": 37})}[shape]()
    E, U = env.num_envs, env.plan.num_ues
    env.reset()
    vals = R.near_cents_and_ties(4)
    rng = np.random.default_rng(11)
    rounds = -(-len(vals) // (E * U))
    pool = np.resize(rng.permutation(vals), rounds * E * U).reshape(rounds, E, U)
    thresholds = R.cent_thresholds()
    scorers = [LayoutScorer(env, float(t)) for t in thresholds]
    for r in range(rounds):
        env.utility_scaled.copy_(torch.from_numpy(pool[r]))
        for sc in scorers:
            sc.update()
    u = pool.transpose(1, 0, 2).reshape(E, rounds * U)
    depth = rounds + -(-U // 32) + 5 + 1
    for t, sc in zip(thresholds, scorers):
        _check_acc(sc.acc.cpu().numpy(), u, t, depth, f"threshold {t!r}")


def _reachable_d2(d2max, side):
    """{d2: (dx, dy)} for every d2 <= d2max that is dx^2 + dy^2 with 0 <= dx, dy < side."""
    out = {}
    for dx in range(side):
        for dy in range(side):
            d2 = dx * dx + dy * dy
            if d2 <= d2max and d2 not in out:
                out[d2] = (dx, dy)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("generic", [False, True])
def test_every_reachable_rate_of_mcomcustom(generic):
    """One env per (UEs on the BS n = 1..7, reachable d2): n - 1 UEs on the BS, a probe UE at distance d2,
    the rest out of range, all standing still for one step.  The rate is round(rate_lut[d2] / n, 2), the
    FP32 utility stays within the documented error of the FP64 one, every cent equals the dump files' cent
    and every threshold count is exact -- on the thread-per-env or the generic step kernel, and (thread-per-env)
    in the fused one-step episode."""
    import torch
    from mobile_env_gan_b200.export import scaled_utility_fp64
    from mobile_env_gan_b200.scenarios import MComCustom
    from mobile_env_gan_b200.scoring import LayoutScorer

    U, B = 7, 10
    probe = MComCustom(config={"num_envs": 32})
    cls = probe.plan.classes[0]
    lut, d2max = np.asarray(cls["rate_lut"], dtype=np.float64), int(cls["d2max"])
    side = int(probe.plan.width)
    reach = _reachable_d2(d2max, side)
    assert len(reach) == 5101 and 2 * (side - 1) ** 2 > d2max
    cases = [(n, d2) for n in range(1, U + 1) for d2 in sorted(reach)]
    assert len(cases) == 35707
    cases += [cases[-1]] * (-len(cases) % 32)  # the thread-per-env kernel takes whole warps of envs
    E = len(cases)
    pos = np.full((E, U, 2), side - 1, dtype=np.int16)
    for e, (n, d2) in enumerate(cases):
        pos[e, : n - 1] = 0
        pos[e, n - 1] = reach[d2]
    env = MComCustom(config={"num_envs": E, "generic_kernel": generic, "autoreset": False})
    assert env.step_kernel_name == ("step_kernel" if generic else "step_tpe_fork_kernel")
    env.reset()
    env.set_station_positions(np.zeros((E, B, 2), dtype=np.int16))  # every live slot on (0, 0): BS 0 serves
    env.set_positions(pos)
    env.inject_waypoints(pos[:, :, None, :])  # the waypoint is the position: nobody moves
    start = env.state_dict()
    thresholds = R.cent_thresholds()
    scorers = [LayoutScorer(env, float(t)) for t in thresholds]
    env.step(0, 0)
    for sc in scorers:
        sc.update()
    assert torch.equal(env.pos, torch.from_numpy(pos).to(env.device))

    n = np.array([c[0] for c in cases])
    d2 = np.array([c[1] for c in cases])
    ue = np.arange(U)[None, :]
    want_rate = np.where(ue < n[:, None] - 1, np.round(lut[0] / n, 2)[:, None], 0.0)
    want_rate = np.where(ue == n[:, None] - 1, np.round(lut[d2] / n, 2)[:, None], want_rate)
    assert np.array_equal(env.assoc.cpu().numpy(), np.where(ue < n[:, None], 0, -1))
    assert np.array_equal(env.rate.cpu().numpy(), want_rate)

    util = env.utility_scaled.cpu().numpy()
    rates, inv = np.unique(want_rate, return_inverse=True)
    u64 = np.array([scaled_utility_fp64(float(r), *DEFAULT_UTILITY) for r in rates])[inv.reshape(E, U)]
    err = float(np.max(np.abs(util.astype(np.float64) - u64)))
    bound = R.device_utility_error_bound(DEFAULT_UTILITY, 100.0)
    print(f"max |FP32 utility - FP64| over {len(rates)} rates: {err:.3e} (bound {bound:.3e}, "
          f"tie margin {R.tie_margin(DEFAULT_UTILITY, 100.0):.3e})")
    assert err <= bound
    assert np.array_equal(R.cents(util), np.rint(u64 * 100))
    assert int(np.sum(np.rint(u64 * 100) == 10)) >= 197  # QoE 0.10 really occurs

    for t, sc in zip(thresholds, scorers):
        _check_acc(sc.acc.cpu().numpy(), util, t, 7, f"threshold {t!r}")
    if not generic:  # the same step as a fused episode of one step (ROLLOUT branch of the kernel)
        for t, sc in zip(thresholds, scorers):
            env.load_state_dict(start)
            acc = torch.zeros_like(sc.acc)
            before = env.launch_count
            env.rollout(1, qoe_acc=acc, threshold=float(t))
            assert env.launch_count - before == 1
            assert torch.equal(acc, sc.acc), t


def _episode_env(case, autoreset, E):
    from mobile_env_gan_b200.scenarios import MComCustom, MComLarge, MComMedium, MComSmall

    if case.startswith("custom"):
        M = 4 if case == "custom-m4" else 1
        return MComCustom(config={"num_envs": E, "autoreset": autoreset, "num_trajectories": M})
    cls = {"small": MComSmall, "medium": MComMedium, "large": MComLarge}[case]
    return cls(config={"num_envs": E, "autoreset": autoreset, "mode": "fork", "ue": {"velocity": 7.5}})


@pytest.mark.gpu
@pytest.mark.parametrize("case,autoreset", [
    ("custom", False), ("custom", True),  # step_tpe_fork_kernel<7, 10, ROLLOUT>
    ("small", True), ("small", False),    # <5, 3, ROLLOUT, SHARED>
    ("medium", True), ("medium", False),  # <15, 4, ROLLOUT, SHARED>
    ("large", True),                      # no fused kernel: steps + qoe_accumulate_kernel
    ("custom-m4", True),                  # four trajectories per layout, pooled
])
def test_episode_statistics_and_result_match_the_fp64_restatement(case, autoreset):
    """A whole episode started mid-episode, at thresholds {0, 0.1, 0.3, -0.05, 0.5}: the accumulators
    equal the restatement of the recorded utility series, whose cents equal those of the recorded FP64
    rates through ``export.scaled_utility_fp64`` (the dump files); ``result()`` is within the bound derived
    for FP32 (below 1e-5) of FP64 ``qoeValue`` and ``best(k)`` is the FP64 top k wherever the gaps allow."""
    import torch
    from mobile_env_gan_b200.export import scaled_utility_fp64
    from mobile_env_gan_b200.scoring import LayoutScorer

    E = 2048
    env = _episode_env(case, autoreset, E)
    U, M, T = env.plan.num_ues, env.plan.num_trajectories, 30 if autoreset else env.plan.ep_time - 1
    env.reset()
    env.step(0, 0)  # start mid-episode
    start = env.state_dict()
    fused = case != "large"
    series = None
    for t in EPISODE_THRESHOLDS:
        env.load_state_dict(start)
        sc = LayoutScorer(env, t)
        before = env.launch_count
        rec = sc.run_episode(T, record=("rate", "utility"))
        assert env.launch_count - before == (1 if fused else 2 * T)
        if series is None:
            series = {k: v.cpu().numpy() for k, v in rec.items()}
            util, rate = series["utility"], series["rate"]  # [T, E, U]
            # the cents of the kernels' FP32 utility are those of the dump files' FP64 QoE
            rates, inv = np.unique(rate, return_inverse=True)
            up = env.config["utility_params"]
            u64 = np.array([scaled_utility_fp64(float(r) if r > 0 else 0.0, up["lower"], up["upper"],
                                                tuple(up["coeffs"])) for r in rates])[inv.reshape(rate.shape)]
            assert np.array_equal(R.cents(util), np.rint(u64 * 100))
            u = util.transpose(1, 0, 2).reshape(E // M, M * T * U)  # a layout's M rows side by side
            assert len(np.unique(R.cents(util))) > 20  # the episode really spreads over the cents
        else:
            for k, v in rec.items():
                assert np.array_equal(v.cpu().numpy(), series[k]), k
        depth = T + -(-U // 32) + 5 + 1 + (M - 1)
        exact, (e1, e2) = _check_acc(sc.pooled().cpu().numpy(), u, t, depth, f"{case} threshold {t}")
        ref = R.qoe_value(*exact)
        eb = R.result_error_bound(ref, exact[3], e1, e2)
        got = {k: v.cpu().numpy().astype(np.float64) for k, v in sc.result().items()}
        for key in ref:
            assert np.all(np.abs(got[key] - ref[key]) <= eb[key]), (key, np.max(np.abs(got[key] - ref[key]) - eb[key]))
        assert float(np.max(eb["Score"])) < 1e-5
        # best(k): the FP64 order wherever the FP64 gaps exceed what FP32 may move two scores
        k = 16
        idx, top = (v.cpu().numpy() for v in sc.best(k))
        order = np.argsort(-ref["Score"], kind="stable")
        s = ref["Score"][order]
        tol = 2 * float(np.max(eb["Score"]))
        assert np.all(np.abs(ref["Score"][idx] - s[:k]) <= tol)
        for i in range(k):
            clear = (i == 0 or s[i - 1] - s[i] > tol) and s[i] - s[i + 1] > tol
            if clear:
                assert idx[i] == order[i], (i, idx[i], order[i])
