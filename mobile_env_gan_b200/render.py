"""Palette and default style of the map-panel frames drawn by ``mbe_render`` (DESIGN.md section 9).

The colours live here and only here: ``MComCore.render_frames`` passes them to the kernel, and the
test restatement (``oracle/render_ref.py``) imports them from this module."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib

# palette rows (include/mbe.h mbe_render_style)
BACKGROUND, COVERAGE, BS, UNCONNECTED, RAMP = 0, 1, 4, 5, 6
PALETTE_SIZE = _lib.RENDER_PALETTE
DEFAULT_SIZE = (256, 256)  # (height, width) in pixels
UE_RADIUS, BS_HALF, LINE_WIDTH = 3, 4, 1
MAX_STYLE_PX = 64  # MBE_RENDER_MAX_STYLE_PX


def _ramp() -> np.ndarray:
    """256 utility colours from red (u = -1) over yellow (u = 0) to green (u = 1), integer interpolation."""
    stops = np.array([(215, 48, 39), (254, 224, 139), (26, 152, 80)], dtype=np.int64)
    i = np.arange(256, dtype=np.int64)
    lo = np.minimum(i // 128, 1)
    f = i - 128 * lo  # 0..127 inside each half (i = 255 ends at 127/128 of the way to green)
    return ((stops[lo] * (128 - f[:, None]) + stops[lo + 1] * f[:, None] + 64) // 128).astype(np.uint8)


PALETTE = np.concatenate([
    np.array([(255, 255, 255),                                   # background
              (222, 235, 247), (198, 219, 239), (158, 202, 225),  # covered by 1 / 2 / >= 3 BSs
              (33, 33, 33),                                       # BS square
              (150, 150, 150)], dtype=np.uint8),                  # UE without a connection
    _ramp(),
])
assert PALETTE.shape == (PALETTE_SIZE, 3)


def ramp_index(utility) -> np.ndarray:
    """Ramp row of a connected UE: clamp(floor((u + 1) * 128), 0, 255) in float32 (the add rounded on its own,
    the multiply by 128 exact).  NaN maps to 0, as in the kernel."""
    v = np.floor((np.asarray(utility, dtype=np.float32) + np.float32(1.0)) * np.float32(128.0))
    return np.where(v >= 255, 255, np.where(v > 0, v, 0)).astype(np.int64)


def style(size=None, ue_radius=UE_RADIUS, bs_half=BS_HALF, line_width=LINE_WIDTH) -> "_lib.RenderStyle":
    """``mbe_render_style`` for a frame of ``size`` = (height, width) pixels (default ``DEFAULT_SIZE``)."""
    h, w = DEFAULT_SIZE if size is None else size
    st = _lib.RenderStyle()
    st.height, st.width = int(h), int(w)
    st.ue_radius, st.bs_half, st.line_width = int(ue_radius), int(bs_half), int(line_width)
    C.memmove(st.palette, PALETTE.tobytes(), PALETTE.nbytes)
    return st
