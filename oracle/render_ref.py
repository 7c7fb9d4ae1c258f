"""Numpy restatement of the map-panel frame (DESIGN.md section 9), vectorised over pixels.

Test infrastructure only: the product never imports it.  Every geometric test is integer arithmetic
(int64 here), so a frame of the CUDA kernel ``mbe_render`` must equal this one byte for byte.  Palette
and default style come from ``mobile_env_gan_b200.render``; ``d2max`` per link class from
``Channel.fold`` (the folded classes of ``MComCore.build_plan``)."""
from __future__ import annotations

import numpy as np

from mobile_env_gan_b200 import render as R


def sample_points(H, W, Wm, Hm):
    """Integer map point sampled by every pixel: xs [W] per column, ys [H] per row (row 0 = top)."""
    j = np.arange(W, dtype=np.int64)
    i = np.arange(H, dtype=np.int64)
    return ((2 * j + 1) * Wm) // (2 * W), ((2 * (H - 1 - i) + 1) * Hm) // (2 * H)


def to_pixel(xy, H, W, Wm, Hm):
    """Pixel (cx, cy) of integer map points xy [..., 2], clamped into the frame."""
    xy = np.asarray(xy, dtype=np.int64)
    cx = np.clip((xy[..., 0] * W) // Wm, 0, W - 1)
    cy = np.clip(H - 1 - (xy[..., 1] * H) // Hm, 0, H - 1)
    return cx, cy


def on_segment(px, py, ax, ay, bx, by, w):
    """4 dist^2(P, segment AB) <= w^2 in exact integer arithmetic (int64): endpoint distances when the
    projection of P falls outside the segment, else 4 cross^2 <= w^2 |B - A|^2."""
    px, py, ax, ay, bx, by = (np.asarray(v, dtype=np.int64) for v in (px, py, ax, ay, bx, by))
    dx, dy, rx, ry = bx - ax, by - ay, px - ax, py - ay
    len2 = dx * dx + dy * dy
    t = dx * rx + dy * ry
    cross = dx * ry - dy * rx
    da = 4 * (rx * rx + ry * ry) <= w * w
    db = 4 * ((px - bx) ** 2 + (py - by) ** 2) <= w * w
    mid = 4 * cross * cross <= w * w * len2
    return np.where(t <= 0, da, np.where(t >= len2, db, mid))


def coverage_counts(xs, ys, bs_xy, d2max):
    """Number of BSs b with (xs - bx)^2 + (ys - by)^2 <= d2max[b] at every sample point -> [H, W]."""
    cnt = np.zeros((len(ys), len(xs)), dtype=np.int64)
    for (bx, by), d2 in zip(np.asarray(bs_xy, dtype=np.int64), d2max):
        if d2 < 0:
            continue
        cnt += ((ys[:, None] - by) ** 2 + (xs[None, :] - bx) ** 2) <= d2
    return cnt


def render_frame(width, height, bs_xy, d2max, ue_pos, conn, utility, size=None, ue_radius=R.UE_RADIUS,
                 bs_half=R.BS_HALF, line_width=R.LINE_WIDTH):
    """One frame uint8 [H, W, 3].

    width, height: the map (int() of them is used); bs_xy [nb, 2]: the LIVE BS slots; d2max [nb]: per slot,
    of the link class (BS class, UE class 0); ue_pos [U, 2]; conn bool [U, nb]: UE u connected to slot b;
    utility [U] float32."""
    H, W = R.DEFAULT_SIZE if size is None else size
    Wm, Hm = int(width), int(height)
    xs, ys = sample_points(H, W, Wm, Hm)
    idx = np.minimum(coverage_counts(xs, ys, bs_xy, d2max), 3)  # 0 = background, 1..3 tints
    py, px = np.mgrid[0:H, 0:W].astype(np.int64)
    bcx, bcy = to_pixel(np.asarray(bs_xy).reshape(-1, 2), H, W, Wm, Hm)
    ucx, ucy = to_pixel(np.asarray(ue_pos).reshape(-1, 2), H, W, Wm, Hm)
    conn = np.asarray(conn, dtype=bool).reshape(len(ucx), len(bcx))
    connected = conn.any(axis=1)
    ue_col = np.where(connected, R.RAMP + R.ramp_index(utility), R.UNCONNECTED)
    for u in range(len(ucx)):  # lines: UE order, then BS order; a later one paints over an earlier one
        for b in np.flatnonzero(conn[u]):
            hit = on_segment(px, py, ucx[u], ucy[u], bcx[b], bcy[b], line_width)
            idx[hit] = ue_col[u]
    for b in range(len(bcx)):
        idx[(np.abs(px - bcx[b]) <= bs_half) & (np.abs(py - bcy[b]) <= bs_half)] = R.BS
    for u in range(len(ucx)):
        idx[(px - ucx[u]) ** 2 + (py - ucy[u]) ** 2 <= ue_radius * ue_radius] = ue_col[u]
    return R.PALETTE[idx]


def link_d2max(plan):
    """d2max per BS slot of a plan: link class (bs_class[b], UE class 0) of the folded classes."""
    nuc = max(1, len(plan.ue_classes))
    bs_class = np.zeros(plan.num_bs, dtype=np.int64) if plan.bs_class is None else plan.bs_class.astype(np.int64)
    return np.array([plan.classes[c * nuc]["d2max"] for c in bs_class], dtype=np.int64)


def render_env_state(plan, width, height, bs_xy, nbs, pos, conn_words, assoc, utility, size=None):
    """Frame of one env from host copies of its state: bs_xy [B, 2], nbs (int or None), pos [U, 2],
    conn_words uint32 [U, MW] (GYM) or None, assoc [U] (FORK) or None, utility [U]."""
    nb = plan.num_bs if nbs is None else int(nbs)
    U = len(pos)
    conn = np.zeros((U, nb), dtype=bool)
    if conn_words is not None:
        words = np.asarray(conn_words, dtype=np.int64).reshape(U, -1) & 0xFFFFFFFF
        for b in range(nb):
            conn[:, b] = (words[:, b // 32] >> (b % 32)) & 1
    else:
        a = np.asarray(assoc)
        for u in range(U):
            if 0 <= a[u] < nb:
                conn[u, a[u]] = True
    return render_frame(width, height, np.asarray(bs_xy)[:nb], link_d2max(plan)[:nb], pos, conn, utility, size=size)
