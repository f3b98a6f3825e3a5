"""ORACLE (test infrastructure, not product code): the injected trail of lfd_submit_injected (include/lfd_b200.h,
lfd_trail) in NumPy float32.  It is the checker of k_inject, not a fallback.

The trail is lfd_b200/synth.py::_add_trail's Gaussian line segment in the same float32 operation order, with the tails
beyond the cut-off dropped: pixel (x, y) gets peak * exp(-0.5 * (d / sigma)**2) added iff 0 <= t <= L and
|d| <= ceil(5 * sigma) + 1, where

    t = (x - x0) * ux + (y - y0) * uy,    d = -(x - x0) * uy + (y - y0) * ux

and ux, uy, L are computed in double from the float32 end points, then rounded to float32.  On end points that are
exact float32 values this is bit-identical to _add_trail wherever both add flux, and it never adds flux outside
_add_trail's bounding box.
"""
import math

import numpy as np


def trail_params(trail):
    """(x0, y0, ux, uy, L, sigma, peak, pad) as float32 scalars (L = 0 for a zero-length trail)."""
    x0, y0 = np.float32(trail["p0"][0]), np.float32(trail["p0"][1])
    x1, y1 = np.float32(trail["p1"][0]), np.float32(trail["p1"][1])
    sigma, peak = np.float32(trail["sigma"]), np.float32(trail["peak"])
    dx, dy = float(x1) - float(x0), float(y1) - float(y0)
    L = float(np.hypot(dx, dy))
    ux, uy = (dx / L, dy / L) if L > 0 else (0.0, 0.0)
    pad = np.float32(math.ceil(5 * float(sigma)) + 1)
    return x0, y0, np.float32(ux), np.float32(uy), np.float32(L), sigma, peak, pad


def _box(x0, y0, ux, uy, L, pad, h, w):
    """Row / column bounds of the rotated rectangle, widened by 2 px (more than the float32 rounding of t and d)."""
    ex, ey = float(ux) * float(L), float(uy) * float(L)
    nx, ny = -float(uy) * float(pad), float(ux) * float(pad)
    xs = [float(x0) + a * ex + b * nx for a in (0, 1) for b in (-1, 1)]
    ys = [float(y0) + a * ey + b * ny for a in (0, 1) for b in (-1, 1)]
    xa, xb = max(int(math.floor(min(xs))) - 2, 0), min(int(math.ceil(max(xs))) + 3, w)
    ya, yb = max(int(math.floor(min(ys))) - 2, 0), min(int(math.ceil(max(ys))) + 3, h)
    return ya, yb, xa, xb


def footprint(shape, trail):
    """(ya, yb, xa, xb, inside, contribution) of one trail: inside is the boolean footprint on rows ya:yb, columns
    xa:xb, contribution the float32 flux it adds there (None when the trail adds nothing)."""
    h, w = shape
    x0, y0, ux, uy, L, sigma, peak, pad = trail_params(trail)
    if L == 0:
        return None
    ya, yb, xa, xb = _box(x0, y0, ux, uy, L, pad, h, w)
    if ya >= yb or xa >= xb:
        return None
    yy, xx = np.mgrid[ya:yb, xa:xb].astype(np.float32)
    t = (xx - x0) * ux + (yy - y0) * uy
    d = -(xx - x0) * uy + (yy - y0) * ux
    inside = (t >= 0) & (t <= L) & (np.abs(d) <= pad)
    prof = np.exp(np.float32(-0.5) * (d / sigma) ** 2)
    return ya, yb, xa, xb, inside, (peak * prof).astype(np.float32)


def render_trails(img, trails):
    """Add ``trails`` (synth's dicts {p0: (x, y), p1: (x, y), sigma, peak}) to the float32 frame ``img`` in place, in
    trail order; returns ``img``."""
    if img.dtype != np.float32:
        raise TypeError("img must be float32")
    for tr in trails:
        fp = footprint(img.shape, tr)
        if fp is None:
            continue
        ya, yb, xa, xb, inside, add = fp
        view = img[ya:yb, xa:xb]
        view[inside] += add[inside]
    return img
