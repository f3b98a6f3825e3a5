"""Test infrastructure, not product code: the injected trail of lfd_submit_injected_shaped (include/lfd_b200.h,
lfd_table) in NumPy float32.  It is the checker of k_inject's tabulated shapes, not a fallback.

It extends oracle/inject_ref.py (the Gaussian trail, used here unchanged) with ``tables``, a list of
``(lo, hi, samples)`` (the pool of lfd_set_trail_tables).  A trail's ``"profile"`` key selects a tabulated
cross-section on [lo, hi] and its ``"lightcurve"`` key a light curve over 0 <= t <= L; -1 or absent means the Gaussian
and a constant 1.  The footprint is 0 <= t <= L and lo <= d <= hi, and the pixel gets fl(fl(peak * P) * A) added, with P
and A linearly interpolated in float32 round-to-nearest steps.  Without shape keys a trail is oracle/inject_ref.py's.
"""
import numpy as np

from oracle.inject_ref import _box, trail_params


def _lerp(samples, u, inside):
    """samples[i] + f * (samples[i+1] - samples[i]), i = min(trunc(u), n - 2), f = u - i, in float32 (u >= 0 inside)."""
    a = np.asarray(samples, np.float32)
    u = np.where(inside, u, np.float32(0))
    i = np.minimum(np.trunc(u).astype(np.int64), len(a) - 2)
    f = u - i.astype(np.float32)
    return a[i] + f * (a[i + 1] - a[i])


def footprint(shape, trail, tables=None):
    """(ya, yb, xa, xb, inside, contribution) of one trail: inside is the boolean footprint on rows ya:yb, columns
    xa:xb, contribution the float32 flux it adds there (None when the trail adds nothing)."""
    h, w = shape
    prof_i, lc_i = int(trail.get("profile", -1)), int(trail.get("lightcurve", -1))
    if prof_i >= 0:
        trail = dict(trail, sigma=1.0)            # a tabulated profile ignores sigma
    x0, y0, ux, uy, L, sigma, peak, pad = trail_params(trail)
    if L == 0:
        return None
    if prof_i >= 0:
        lo, hi, psmp = tables[prof_i]
        dlo, dhi = np.float32(lo), np.float32(hi)
        pad = max(abs(dlo), abs(dhi))
    else:
        dlo, dhi = -pad, pad
    ya, yb, xa, xb = _box(x0, y0, ux, uy, L, pad, h, w)
    if ya >= yb or xa >= xb:
        return None
    yy, xx = np.mgrid[ya:yb, xa:xb].astype(np.float32)
    t = (xx - x0) * ux + (yy - y0) * uy
    d = -(xx - x0) * uy + (yy - y0) * ux
    inside = (t >= 0) & (t <= L) & (d >= dlo) & (d <= dhi)
    if prof_i >= 0:
        inv = np.float32((len(psmp) - 1) / (float(dhi) - float(dlo)))
        prof = _lerp(psmp, (d - dlo) * inv, inside)
    else:
        prof = np.exp(np.float32(-0.5) * (d / sigma) ** 2)
    add = (peak * prof).astype(np.float32)
    if lc_i >= 0:
        asmp = tables[lc_i][2]
        c = np.float32((len(asmp) - 1) / float(L))
        add = add * _lerp(asmp, t * c, inside)
    return ya, yb, xa, xb, inside, add


def render_trails(img, trails, tables=None):
    """Add ``trails`` (synth's dicts {p0: (x, y), p1: (x, y), sigma, peak}, optionally with ``"profile"`` and
    ``"lightcurve"`` indices into ``tables``) to the float32 frame ``img`` in place, in trail order; returns ``img``."""
    if img.dtype != np.float32:
        raise TypeError("img must be float32")
    for tr in trails:
        fp = footprint(img.shape, tr, tables)
        if fp is None:
            continue
        ya, yb, xa, xb, inside, add = fp
        view = img[ya:yb, xa:xb]
        view[inside] += add[inside]
    return img
