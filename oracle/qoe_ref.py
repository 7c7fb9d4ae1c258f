"""FP64 restatement of the QoE statistics behind the layout score (DESIGN.md sections 2 and 10.1,
include/mbe.h ``mbe_accumulate_qoe`` and ``mbe_rollout``).

Test infrastructure only: the product never imports it.  The contract it restates:

* the cent of a QoE value u (FP32, as the kernels hold it) is k = the exact half-even rounding of
  u * 100 -- ``np.rint(float64(u) * 100)``, exact because the product of a float32 and 100 fits 53 bits;
* the two-decimal value is q = float32(k / 100), and it is low QoE when q < float32(threshold).

That is Python's ``round(u, 2) < t`` for every cent-valued t; a threshold within one float32 ulp of a
cent acts as that cent.  The score (chooseBaseStation.ipynb cell 5 ``qoeValue``) is
``mean - 0.1 * var - 10 * P(low)`` over all values of an epoch, here in FP64 over k / 100."""
from __future__ import annotations

import math

import numpy as np

F32_EPS = 2.0**-24  # unit roundoff of FP32


def cents(u):
    """The cent k (FP64 integer values) of FP32 QoE values u."""
    return np.rint(np.asarray(u, dtype=np.float32).astype(np.float64) * 100)


def cent_value(k):
    """The two-decimal value float32(k / 100) the kernels add up."""
    return (np.asarray(k, dtype=np.float64) / 100).astype(np.float32)


def is_low(k, threshold):
    """The low-QoE predicate float32(k / 100) < float32(threshold)."""
    return cent_value(k) < np.float32(threshold)


def accumulate(u, threshold, axis=-1):
    """The four accumulators (sum q, sum q^2, #low, #values) in FP64 over ``axis`` of FP32 QoE values u,
    with q = k / 100 in FP64 (the notebook's values)."""
    k = cents(u)
    q = k / 100
    low = is_low(k, threshold)
    n = np.full(q.sum(axis=axis).shape, q.shape[axis], dtype=np.float64)
    return q.sum(axis=axis), (q * q).sum(axis=axis), low.sum(axis=axis).astype(np.float64), n


def qoe_value(s1, s2, low, n, weights=(1.0, 0.1, 10.0)):
    """``qoeValue`` from the accumulators, in FP64: a dict with ``LayoutScorer.result()``'s keys."""
    s1, s2, low, n = (np.asarray(v, dtype=np.float64) for v in (s1, s2, low, n))
    mean = s1 / n
    var = s2 / n - mean * mean
    p = low / n
    w1, w2, w3 = weights
    return {"Average QoE": mean, "QoE Variance": var, "Low QoE Proportion": p,
            "Score": w1 * mean - w2 * var - w3 * p}


def sum_error_bound(abs_sum, depth, rel_term=F32_EPS):
    """|FP32 sum - exact sum| for terms that carry a relative error ``rel_term`` each and pass through at
    most ``depth`` FP32 additions on the way into the sum (gamma_depth, Higham 2002, section 4.2)."""
    g = depth * F32_EPS / (1 - depth * F32_EPS)
    return (rel_term + g) * (1 + g) * np.asarray(abs_sum, dtype=np.float64)


def result_error_bound(ref, n, e_s1, e_s2, weights=(1.0, 0.1, 10.0)):
    """Per key, the largest distance of ``LayoutScorer.result()`` (FP32 arithmetic on FP32 accumulators that
    lie within e_s1 / e_s2 of the exact sums, exact counts) from ``qoe_value`` ``ref``."""
    u = F32_EPS
    mean, var, p = (np.abs(ref[k]) for k in ("Average QoE", "QoE Variance", "Low QoE Proportion"))
    m2 = var + mean * mean  # s2 / n
    e_mean = e_s1 / n + 2 * u * mean
    e_var = e_s2 / n + 2 * u * m2 + 2 * (mean + e_mean) * e_mean + 2 * u * mean * mean + 2 * u * var
    e_p = 2 * u * p
    w1, w2, w3 = (abs(w) for w in weights)
    e_score = w1 * e_mean + w2 * e_var + w3 * e_p + 4 * u * (w1 * mean + w2 * var + w3 * p) + 4 * u * w3 * e_p
    return {"Average QoE": e_mean, "QoE Variance": e_var, "Low QoE Proportion": e_p, "Score": e_score}


def scaled_utility_fp64_array(rate, lower, upper, coeffs):
    """``export.scaled_utility_fp64`` over an array of rates (np.log of arrays may differ from the scalar
    path in the last bit, which no margin below depends on)."""
    w1, w2, w3 = coeffs
    rate = np.asarray(rate, dtype=np.float64)
    u = np.where(rate <= 0.0, lower, np.clip(w1 * np.log(w2 + np.maximum(rate, 1e-300)) / np.log(w3), lower, upper))
    return 2 * (u - lower) / (upper - lower) - 1


def saturation_rate(utility_params, rate_max):
    """rate_max, capped at the two-decimal rate from which an increasing utility is clipped to ``upper``
    (every larger rate has the scaled utility 1 exactly)."""
    lower, upper, (w1, w2, w3) = utility_params
    if w1 / np.log(w3) > 0:
        rate_max = min(rate_max, math.ceil((w3 ** (upper / w1) - w2) * 100 + 1) / 100)
    return rate_max


def tie_margin(utility_params, rate_max):
    """The smallest distance, in QoE units, from the FP64 scaled utility of a two-decimal rate in
    (0, rate_max] to a half-cent tie.  When the kernels' FP32 utility error stays below it, every kernel
    cent equals the FP64 cent of the dump files; parameters with a smaller margin may give other cents."""
    lower, upper, coeffs = utility_params
    rate_max = saturation_rate(utility_params, rate_max)
    rates = np.arange(1, int(round(rate_max * 100)) + 1, dtype=np.float64) / 100
    x = scaled_utility_fp64_array(rates, lower, upper, coeffs) * 100
    return float(np.min(np.abs(x - (np.floor(x) + 0.5)))) / 100


def device_utility_error_bound(utility_params, rate_max):
    """Bound on |FP32 scaled utility of the kernels - FP64 scaled utility| for rates in (0, rate_max]
    (``scaled_utility`` in mbe_device.cuh): lg2.approx.ftz.f32 within 2^-22 * max(1, |log2 x|) of log2 x,
    the rate rounded to FP32, and a few FP32 roundings of values up to max(|lower|, |upper|, upper - lower)."""
    lower, upper, (w1, w2, w3) = utility_params
    c = abs(w1 / np.log2(w3))
    lg = max(abs(np.log2(w2 + 0.01)), abs(np.log2(w2 + saturation_rate(utility_params, rate_max))), 1.0)
    e_lg2 = 2.0**-22 * lg + F32_EPS / np.log(2)
    scale = 2.0 / (upper - lower)
    big = max(abs(lower), abs(upper), upper - lower)
    return scale * (c * e_lg2 + 3 * F32_EPS * big) + 3 * F32_EPS


def near_cents_and_ties(ulps=64):
    """Every float32 within +-ulps of each of the 201 cents k / 100 and 200 half-cent ties (k + 0.5) / 100
    in [-1, 1], plus +-0 and +-1: the inputs on which a cent rounding or a threshold test goes wrong."""
    k = np.arange(-100, 101)
    centers = np.concatenate([k / 100, (k[:-1] + 0.5) / 100]).astype(np.float32)
    bits = centers.view(np.int32).astype(np.int64)
    step = np.arange(-ulps, ulps + 1)
    # float32 bit patterns are monotone within one sign; walk across zero through the signed ordering
    order = np.where(bits < 0, -(bits & 0x7FFFFFFF), bits)[:, None] + step[None, :]
    pat = np.where(order < 0, (-order) | np.int64(0x80000000), order).astype(np.uint32)
    vals = pat.view(np.float32).ravel()
    extra = np.array([0.0, -0.0, 1.0, -1.0], dtype=np.float32)
    return np.unique(np.concatenate([vals, extra]).view(np.uint32)).view(np.float32)


def cent_thresholds():
    """Every cent threshold k / 100 in [-1, 1] as float32, plus -0.0, a half cent and +-1.5."""
    return np.concatenate([cent_value(np.arange(-100, 101)), np.array([-0.0, 0.005, 1.5, -1.5], dtype=np.float32)])
