"""Injection and recovery: what fraction of trails of a given brightness, width, angle and length the bright + dim
passes find.  Synthetic trails (synth's dicts ``{p0: (x, y), p1: (x, y), sigma, peak}``, the Gaussian line segment of
include/lfd_b200.h ``lfd_trail``) are added to resident real frames on the device (lfd_set_base /
lfd_submit_injected), so a campaign that reuses a few dozen frames thousands of times never sends pixels over the host
link."""
import math

import numpy as np

from . import _lib

__all__ = ["trail_line", "recovery", "RECOVERY_DTYPE"]

_T = _lib.MAX_INJECT_TRAILS
RECOVERY_DTYPE = np.dtype([
    ("base", "<i4"), ("ntrails", "<i4"),
    ("x0", "<f4", (_T,)), ("y0", "<f4", (_T,)), ("x1", "<f4", (_T,)), ("y1", "<f4", (_T,)),
    ("sigma", "<f4", (_T,)), ("peak", "<f4", (_T,)),
    ("detected", "?"), ("pass", "<i4"), ("status", "<i4"), ("rho", "<f4"), ("theta", "<f4"),
    ("base_detected", "?"), ("recovered", "<i4")])


def trail_line(trail, shape):
    """(rho, theta) of the injected segment's line in cv2.HoughLines' normal form, x cos(theta) + y' sin(theta) = rho,
    in the flipped frame the passes see (y' = H - 1 - y), with theta in [0, pi) and a signed rho.  (nan, nan) for a
    zero-length trail."""
    h = shape[0]
    x0, y0 = float(trail["p0"][0]), float(h - 1 - trail["p0"][1])
    x1, y1 = float(trail["p1"][0]), float(h - 1 - trail["p1"][1])
    if x0 == x1 and y0 == y1:
        return math.nan, math.nan
    theta = math.fmod(math.atan2(y1 - y0, x1 - x0) + 1.5 * math.pi, math.pi)   # the normal of the direction, mod pi
    if theta >= math.pi:
        theta -= math.pi
    return x0 * math.cos(theta) + y0 * math.sin(theta), theta


def _first_match(rho, theta, lines, theta_tol, rho_tol):
    """Index of the first (rho_true, theta_true) the detected line matches, or -1.  Across the theta = 0 / pi wrap the
    same line has the opposite rho."""
    for i, (rt, tt) in enumerate(lines):
        for k in (-1, 0, 1):
            if abs(theta - tt - k * math.pi) <= theta_tol and abs(rho - (-rt if k else rt)) <= rho_tol:
                return i
    return -1


def recovery(frames, rects, injections, params_bright=None, params_dim=None, device=0, batch=64,
             theta_tol=np.deg2rad(2), rho_tol=None):
    """Run every injection and every base without a trail; one RECOVERY_DTYPE row per injection.

    ``frames``: (n_base, H, W) un-flipped float32 bases; ``rects``: their star rectangles (lfd_submit's convention, one
    array per base) or None; ``injections``: a sequence of ``(base_index, [trail, ...])`` with at most 16 trails each.

    A row holds the base, the injected trails (NaN past ``ntrails``), the device verdict of the injected frame
    (``detected``, ``pass``, ``status``, and ``rho``, ``theta`` = equhough[0][0] of the detecting pass), whether the base
    alone was detected, and ``recovered``: the index of the first injected trail the detected line matches, else -1.  A
    line matches a trail when its theta differs from ``trail_line``'s by at most ``theta_tol`` modulo pi and its rho by
    at most ``rho_tol`` (with rho's sign flipped across the theta = 0 / pi wrap).  ``rho_tol`` defaults to the detecting
    pass's ``houghMethod``, one rho bin of its Hough transform; ``theta_tol`` defaults to 2 degrees, two theta bins.
    The reason for both: on the oracle at houghMethod 20, the detected equhough[0][0] of all 15 detected synth
    ``trail`` / ``trail_var`` frames (of 16) lay within 0.95 degrees and 11.1 px of the injected segment's line, inside
    both defaults; the Hough quantisation itself is one rho bin and one theta bin.

    A frame whose work lists overflow (``status & FRAME_OVERFLOW``) has no valid verdict: it is reported in ``status``
    with ``recovered`` = -1 and not retried on a larger handle.  Two handles alternate, so the host stages one batch
    while the device runs the other."""
    from .detecttrails import default_params
    pb0, pd0, _ = default_params()
    pb = pb0 if params_bright is None else params_bright
    pd = pd0 if params_dim is None else params_dim
    frames = np.ascontiguousarray(frames, np.float32)
    nb, H, W = frames.shape
    jobs = [(b, []) for b in range(nb)] + [(int(b), list(ts)) for b, ts in injections]
    for b, ts in jobs:
        if not 0 <= b < nb:
            raise ValueError("base index %d out of range" % b)
        if len(ts) > _T:
            raise ValueError("at most %d trails per injection" % _T)
    B = max(1, min(int(batch), len(jobs)))
    chunks = [range(i, min(i + B, len(jobs))) for i in range(0, len(jobs), B)]
    res = [None] * len(jobs)
    hs = []
    try:
        for _ in range(2):
            h = _lib.Handle(H, W, max_batch=B, device=device)
            hs.append(h)
            h.set_params(pb, pd)
            h.set_base(frames, rects)

        def submit(k):
            hs[k & 1].submit_injected([jobs[i][0] for i in chunks[k]], [jobs[i][1] for i in chunks[k]])

        def collect(k):
            r = hs[k & 1].wait_array()
            for j, i in enumerate(chunks[k]):
                res[i] = r[j]

        submit(0)
        for k in range(1, len(chunks)):
            submit(k)
            collect(k - 1)
        collect(len(chunks) - 1)
    finally:
        for h in hs:
            h.close()

    out = np.zeros(len(jobs) - nb, RECOVERY_DTYPE)
    hough = (float(pb["houghMethod"]), float(pd["houghMethod"]))
    for row, (b, ts), r in zip(out, jobs[nb:], res[nb:]):
        row["base"], row["ntrails"] = b, len(ts)
        for f in ("x0", "y0", "x1", "y1", "sigma", "peak"):
            row[f] = np.nan
        if ts:
            arr = _lib.Handle.trails_array(ts)
            for f in ("x0", "y0", "x1", "y1", "sigma", "peak"):
                row[f][:len(ts)] = arr[f]
        row["detected"], row["pass"], row["status"] = bool(r["detected"]), r["pass_"], r["status"]
        row["rho"], row["theta"] = r["rho"], r["theta"]
        row["base_detected"] = bool(res[b]["detected"])
        row["recovered"] = -1
        if r["detected"] and not (r["status"] & _lib.FRAME_OVERFLOW):
            rt = hough[r["pass_"]] if rho_tol is None else float(rho_tol)
            row["recovered"] = _first_match(float(r["rho"]), float(r["theta"]), [trail_line(t, (H, W)) for t in ts],
                                            float(theta_tol), rt)
    return out
