"""Numpy restatement of the layout maps (DESIGN.md section 10.2, include/mbe.h ``mbe_layout_map``).

Test infrastructure only: the product never imports it, and it imports nothing of the product.  Every
geometric decision is int64 arithmetic and every rate FP64, so the kernel's coverage, serving BS, area and
counts must equal these exactly; the cents are the FP64 cents of ``oracle/qoe_ref.py``, which the kernel's
FP32 cents equal wherever the utility's tie margin exceeds the device error bound (the default utility)."""
from __future__ import annotations

import math

import numpy as np

from oracle import qoe_ref

STATS = ("points", "covered", "overlap", "sum_k", "sum_k2", "low")


def grid(width, height, stride):
    """Grid coordinates xs [GX], ys [GY]: multiples of stride in [0, ceil(width) - 1] x [0, ceil(height) - 1]."""
    xm, ym = math.ceil(width) - 1, math.ceil(height) - 1
    return np.arange(0, xm + 1, stride, dtype=np.int64), np.arange(0, ym + 1, stride, dtype=np.int64)


def k_low(threshold):
    """The cut of the low-QoE test: cent k is low iff k < k_low (101 when every cent is low)."""
    ks = np.arange(-100, 101)
    ok = ~qoe_ref.is_low(ks, threshold)
    return int(ks[ok][0]) if ok.any() else 101


def shared_rate(rate_lut, load):
    """round(rate_lut[d2] / load, 2) per d2 in FP64, as mbe_create folds its rate table."""
    return np.rint(np.asarray(rate_lut, dtype=np.float64) / load * 100.0) / 100.0


def cents_of_rates(rate, utility):
    """FP64 cents of the scaled utility of rates; utility = (lower, upper, w1, w2, w3)."""
    lower, upper, w1, w2, w3 = utility
    return np.rint(qoe_ref.scaled_utility_fp64_array(rate, lower, upper, (w1, w2, w3)) * 100).astype(np.int64)


def env_map(xs, ys, bs_xy, nb, d2max, cent_tabs, threshold):
    """One env's map.  bs_xy [B, 2] the slots, of which the first clamp(nb, 0, B) are live, d2max [B] per slot
    (-1: never connectable), cent_tabs[b] the cent per d2 of slot b's link class (``cents_of_rates`` of
    ``shared_rate``).  Returns coverage uint8, serving int8, qoe int8 [GY, GX], stats int64 [6], area int64 [B]."""
    bs = np.asarray(bs_xy, dtype=np.int64).reshape(-1, 2)
    B = bs.shape[0]
    nb = min(max(int(nb), 0), B)
    X, Y = np.meshgrid(xs, ys)  # row j is y = ys[j]
    px, py = X.ravel(), Y.ravel()
    d2max = np.asarray(d2max, dtype=np.int64)[:nb]
    d2 = (px[:, None] - bs[None, :nb, 0]) ** 2 + (py[:, None] - bs[None, :nb, 1]) ** 2
    conn = d2 <= d2max[None, :]
    cov = conn.sum(axis=1)
    key = np.where(conn, d2, np.iinfo(np.int64).max)
    serving = np.where(cov > 0, np.argmin(key, axis=1) if nb else -1, -1)  # argmin: the lowest slot of a tie
    k = np.full(px.shape, -100, dtype=np.int64)
    area = np.zeros(B, dtype=np.int64)
    for b in range(nb):
        sel = serving == b
        k[sel] = np.asarray(cent_tabs[b])[d2[sel, b]]
        area[b] = sel.sum()
    stats = np.array([px.size, (cov >= 1).sum(), (cov >= 2).sum(), k.sum(), (k * k).sum(), (k < k_low(threshold)).sum()],
                     dtype=np.int64)
    shape = (len(ys), len(xs))
    return (np.minimum(cov, 255).astype(np.uint8).reshape(shape), serving.astype(np.int8).reshape(shape),
            k.astype(np.int8).reshape(shape), stats, area)


def empty_map(xs, ys, B):
    """The map of an env id outside the handle's range."""
    shape = (len(ys), len(xs))
    return (np.zeros(shape, np.uint8), np.full(shape, -1, np.int8), np.full(shape, -128, np.int8),
            np.zeros(6, np.int64), np.zeros(B, np.int64))


def result(stats, weights=(1.0, 0.1, 10.0)):
    """The statistics keys of ``LayoutMap.result`` in FP64 from stats [..., 6]."""
    pts, cov, ovl, sk, sk2, low = (np.asarray(stats, dtype=np.float64)[..., i] for i in range(6))
    mean = sk / (100 * pts)
    var = sk2 / (10000 * pts) - mean * mean
    p = low / pts
    w1, w2, w3 = weights
    return {"Average QoE": mean, "QoE Variance": var, "Low QoE Proportion": p,
            "Score": w1 * mean - w2 * var - w3 * p, "Coverage": cov / pts, "Overlap": ovl / pts}
