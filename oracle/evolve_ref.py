"""Numpy restatement of one layout-evolution generation (DESIGN.md section 10).

Test infrastructure only: the product never imports it.  Every decision is integer or FP64 arithmetic on
Philox words (``mbe_oracle.philox4x32``), so ``mbe_evolve_layouts`` must produce these children bit for
bit.  Written per child, like the kernel's thread, for readability over speed."""
from __future__ import annotations

import math

import numpy as np

from oracle.mbe_oracle import philox4x32

PURPOSE_EVOLVE = 3


def umulhi(r, n):
    return (int(r) * int(n)) >> 32


def coin(r, p):
    return float(r) * 2.0**-32 < p


def coord_range(width, height):
    """Inclusive [0, XM] x [0, YM]: the values philox_point draws on a width x height map."""
    return math.ceil(width) - 1, math.ceil(height) - 1


def new_point(rx, ry, width, height):
    if width == math.floor(width) and height == math.floor(height):
        return umulhi(rx, int(width)), umulhi(ry, int(height))
    return int(float(rx) * 2.0**-32 * width), int(float(ry) * 2.0**-32 * height)


def _key(fit):
    return -math.inf if math.isnan(fit) else fit


def tournament(words, fitness, T):
    E = len(fitness)
    best = umulhi(words[0], E)
    for j in range(1, T):
        c = umulhi(words[j], E)
        f, bf = _key(fitness[c]), _key(fitness[best])
        if f > bf or (f == bf and c < best):
            best = c
    return best


def evolve(parent_xy, parent_nbs, fitness, elite_ids, *, seed, generation, tournament_size, p_cross, p_move,
           step, p_add, p_del, nmin, nmax, width, height, env_offset=0):
    """parent_xy int [E,B,2], parent_nbs int [E], fitness f32 [E], elite_ids int [K] ->
    (child_xy int16 [E,B,2], child_nbs int32 [E])."""
    parent_xy = np.asarray(parent_xy, dtype=np.int64)
    parent_nbs = np.asarray(parent_nbs, dtype=np.int64)
    fitness = np.asarray(fitness, dtype=np.float32)
    elite_ids = np.asarray(elite_ids, dtype=np.int64).reshape(-1)
    E, B, _ = parent_xy.shape
    nmax = min(nmax, B)
    XM, YM = coord_range(width, height)
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    G = (env_offset + np.arange(E, dtype=np.uint64)).astype(np.uint32)
    # every block every child may use: [4 + B, 4 words, E]
    r = np.stack([np.stack(philox4x32(G, generation, k, PURPOSE_EVOLVE, k0, k1)) for k in range(4 + B)])
    child = np.zeros((E, B, 2), dtype=np.int64)
    child_nbs = np.zeros(E, dtype=np.int64)
    span = 2 * step + 1
    for c in range(E):
        if c < len(elite_ids) and 0 <= elite_ids[c] < E:
            child[c] = parent_xy[elite_ids[c]]
            child_nbs[c] = parent_nbs[elite_ids[c]]
            continue
        p1 = tournament(r[0, :, c], fitness, tournament_size)
        cross = coin(r[2, 0, c], p_cross)
        p2 = tournament(r[1, :, c], fitness, tournament_size) if cross else p1
        n = int(min(max(parent_nbs[p1], 0), B))
        row = np.zeros((B, 2), dtype=np.int64)
        for i in range(n):
            w = r[4 + i, :, c]
            src = p2 if cross and i < parent_nbs[p2] and (int(w[0]) >> 31) else p1
            x, y = parent_xy[src, i]
            if coin(w[1], p_move):
                x = min(max(x + umulhi(w[2], span) - step, 0), XM)
                y = min(max(y + umulhi(w[3], span) - step, 0), YM)
            row[i] = x, y
        if coin(r[2, 1, c], p_add) and n < nmax:
            row[n] = new_point(r[3, 0, c], r[3, 1, c], width, height)
            n += 1
        elif coin(r[2, 2, c], p_del) and n > nmin:
            row[umulhi(r[2, 3, c], n)] = row[n - 1]
            n -= 1
        row[n:] = 0
        child[c], child_nbs[c] = row, n
    return child.astype(np.int16), child_nbs.astype(np.int32)
