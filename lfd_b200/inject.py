"""Injection and recovery: what fraction of trails of a given brightness, width, angle and length the bright + dim
passes find.  Synthetic trails (synth's dicts ``{p0: (x, y), p1: (x, y), sigma, peak}``, the Gaussian line segment of
include/lfd_b200.h ``lfd_trail``) are added to resident real frames on the device (lfd_set_base /
lfd_submit_injected), so a campaign that reuses a few dozen frames thousands of times never sends pixels over the host
link.

Trails may also carry tabulated shapes (include/lfd_b200.h ``lfd_table``): a ``"profile"`` key indexes a cross-section
profile and a ``"lightcurve"`` key a brightness along the segment in the ``tables`` passed to ``recovery``.
``defocus_profile`` builds the cross-section of a meteor seen by a telescope focused at infinity."""
import math

import numpy as np

from . import _lib

__all__ = ["trail_line", "recovery", "defocus_profile", "read_injections", "RECOVERY_DTYPE", "INJECTION_DTYPE"]

_T = _lib.MAX_INJECT_TRAILS
RECOVERY_DTYPE = np.dtype([
    ("base", "<i4"), ("ntrails", "<i4"),
    ("x0", "<f4", (_T,)), ("y0", "<f4", (_T,)), ("x1", "<f4", (_T,)), ("y1", "<f4", (_T,)),
    ("sigma", "<f4", (_T,)), ("peak", "<f4", (_T,)),
    ("detected", "?"), ("pass", "<i4"), ("status", "<i4"), ("rho", "<f4"), ("theta", "<f4"),
    ("base_detected", "?"), ("recovered", "<i4")])
# one row of a drop-in run's injection table (DetectTrails(injections=...), read_injections): the frame and the index k
# of the injection in the callable's list instead of a base index, and each trail's table indices (-1 past ntrails)
INJECTION_DTYPE = np.dtype([
    ("run", "<i4"), ("camcol", "<i4"), ("filter", "U1"), ("field", "<i4"), ("k", "<i4"), ("ntrails", "<i4"),
    ("x0", "<f4", (_T,)), ("y0", "<f4", (_T,)), ("x1", "<f4", (_T,)), ("y1", "<f4", (_T,)),
    ("sigma", "<f4", (_T,)), ("peak", "<f4", (_T,)), ("profile", "<i4", (_T,)), ("lightcurve", "<i4", (_T,)),
    ("detected", "?"), ("pass", "<i4"), ("status", "<i4"), ("rho", "<f4"), ("theta", "<f4"),
    ("base_detected", "?"), ("recovered", "<i4")])
_TRAIL_F = ("x0", "y0", "x1", "y1", "sigma", "peak")


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


def _defocus_samples(r_outer, r_inner, seeing_fwhm, step):
    """(d, samples) of defocus_profile before the normalisation to a maximum of 1 (float64)."""
    ro, ri, fw, step = float(r_outer), float(r_inner), float(seeing_fwhm), float(step)
    if not all(math.isfinite(v) for v in (ro, ri, fw, step)) or step <= 0 or fw < 0:
        raise ValueError("r_outer, r_inner, seeing_fwhm and step must be finite, step > 0 and seeing_fwhm >= 0")
    if ro <= 0 and fw == 0:
        raise ValueError("r_outer must be > 0 when there is no seeing")
    if ri < 0 or ri > ro:
        raise ValueError("r_inner must lie in [0, r_outer]")
    sig = fw / (2.0 * math.sqrt(2.0 * math.log(2.0)))
    k = int(math.ceil((max(ro, 0.0) + 4.0 * sig) / step - 1e-9))
    if 2 * k + 1 > _lib.MAX_TABLE_SAMPLES:
        raise ValueError("%d samples exceed %d: use a larger step" % (2 * k + 1, _lib.MAX_TABLE_SAMPLES))
    # with seeing, the convolution runs on a grid 8 times finer than the output, so the smooth result's samples keep
    # the annulus' integral; without seeing the samples are the annulus' point values
    sub = 8 if sig > 0 else 1
    h = step / sub
    kw = int(math.ceil(4.0 * sig / h)) if sig > 0 else 0
    x = np.arange(-(k * sub + kw), k * sub + kw + 1) * h
    if ro > 0:
        a = np.sqrt(np.maximum(ro * ro - x * x, 0.0)) - np.sqrt(np.maximum(ri * ri - x * x, 0.0))
    else:                                       # a point source: the seeing alone
        a = np.zeros_like(x)
        a[k * sub + kw] = 1.0 / h
    if kw:
        g = np.exp(-0.5 * (np.arange(-kw, kw + 1) * h / sig) ** 2)
        a = np.convolve(a, g / g.sum(), mode="valid")[::sub]
    return np.arange(-k, k + 1) * step, 0.5 * (a + a[::-1])     # exactly symmetric


def defocus_profile(r_outer, r_inner=0.0, seeing_fwhm=0.0, step=0.25):
    """Cross-section of a defocused trail as a ``(lo, hi, samples)`` table for ``recovery(..., tables=...)`` and
    Handle.set_trail_tables: the telescope pupil, a uniform annulus of radii ``r_inner`` <= ``r_outer`` px, drawn along
    a line, sqrt(max(ro² - d², 0)) - sqrt(max(ri² - d², 0)), convolved with the seeing, a Gaussian of FWHM
    ``seeing_fwhm`` px (a 2-D Gaussian projects to a 1-D Gaussian of the same sigma).  Samples every ``step`` px on
    ±(ro + 4 sigma), rounded out to the step, float32, normalised to a maximum of 1, so a trail's ``peak`` is the flux
    at the brightest point of the cross-section.  A telescope focused at infinity images each point of a meteor at
    distance D as its pupil of angular diameter aperture / D: a 2.5 m aperture at 100 km subtends 5.2 arcsec, 13 px at
    0.396 arcsec per pixel, so ``r_outer = 6.5``.  Raises ValueError when r_outer <= 0 without seeing, or r_inner is
    outside [0, r_outer]."""
    d, a = _defocus_samples(r_outer, r_inner, seeing_fwhm, step)
    return float(d[0]), float(d[-1]), (a / a.max()).astype(np.float32)


def _first_match(rho, theta, lines, theta_tol, rho_tol):
    """Index of the first (rho_true, theta_true) the detected line matches, or -1.  Across the theta = 0 / pi wrap the
    same line has the opposite rho."""
    for i, (rt, tt) in enumerate(lines):
        for k in (-1, 0, 1):
            if abs(theta - tt - k * math.pi) <= theta_tol and abs(rho - (-rt if k else rt)) <= rho_tol:
                return i
    return -1


def _recovered(r, trails, shape, hough, theta_tol=np.deg2rad(2), rho_tol=None):
    """``recovered`` of a device result ``r`` (an lfd_result row) for the injected ``trails``: the index of the first
    trail its line matches, -1 when undetected, overflowed or unmatched; ``hough`` = the two passes' houghMethod."""
    if not r["detected"] or (r["status"] & _lib.FRAME_OVERFLOW):
        return -1
    rt = hough[r["pass_"]] if rho_tol is None else float(rho_tol)
    return _first_match(float(r["rho"]), float(r["theta"]), [trail_line(t, shape) for t in trails], float(theta_tol), rt)


def check_injections(specs, n_tables):
    """A frame's injections as the ``injections`` callable of DetectTrails returns them, checked: a list of lists of
    at most 16 trail dicts with finite end points and peak, ``sigma`` > 0 for a Gaussian profile, and ``profile`` /
    ``lightcurve`` indices in -1 .. n_tables - 1.  Raises ValueError naming the first bad trail, also for a missing
    key or a value that is not a number."""
    try:
        specs = [list(ts) for ts in specs]
    except TypeError as e:
        raise ValueError("injections must be a list of lists of trail dicts (%s)" % e) from None
    for k, ts in enumerate(specs):
        if len(ts) > _T:
            raise ValueError("injection %d has %d trails, at most %d are allowed" % (k, len(ts), _T))
        for i, t in enumerate(ts):
            where = "injection %d, trail %d" % (k, i)
            try:
                for key in ("profile", "lightcurve"):
                    v = t.get(key, -1)
                    if not isinstance(v, (int, np.integer)) or isinstance(v, bool) or not -1 <= v < n_tables:
                        raise ValueError("%s %r is not a table index in -1 .. %d" % (key, v, n_tables - 1))
                gauss = t["profile"] < 0 if "profile" in t else True
                vals = [t["p0"][0], t["p0"][1], t["p1"][0], t["p1"][1], t["peak"]] + ([t["sigma"]] if gauss else [])
                with np.errstate(over="ignore"):
                    vals = [float(np.float32(v)) for v in vals]
            except (KeyError, IndexError, TypeError, AttributeError, ValueError) as e:
                raise ValueError("%s: %s" % (where, "missing key %s" % e if isinstance(e, KeyError) else e)) from None
            if not all(math.isfinite(v) for v in vals):
                raise ValueError("%s: end points, sigma and peak must be finite in float32" % where)
            if gauss and not vals[5] > 0:
                raise ValueError("%s: a Gaussian trail needs sigma > 0" % where)
    return specs


def _f9(v):
    return "%.9g" % float(np.float32(v))


def format_injection(frame, k, base_detected, trails, r, recovered):
    """One line of the injection table: ``run camcol filter field k base_detected detected pass status rho theta
    recovered ntrails`` then ``x0 y0 x1 y1 sigma peak profile lightcurve`` per trail (end points un-flipped, as given).
    Floats are the float32 values in %.9g, which reads back to the same bits; ``r`` is the injected frame's lfd_result."""
    run, camcol, flt, field = frame
    arr = _lib.Handle.trails_array(trails)
    head = "%d %d %s %d %d %d %d %d %d %s %s %d %d" % (
        run, camcol, flt, field, k, bool(base_detected), bool(r["detected"]), r["pass_"], r["status"], _f9(r["rho"]),
        _f9(r["theta"]), recovered, len(trails))
    body = "".join(" %s %s %s %s %s %s %d %d" % (tuple(_f9(a[f]) for f in _TRAIL_F) + (t.get("profile", -1), t.get("lightcurve", -1)))
                   for a, t in zip(arr, trails))
    return head + body + "\n"


def read_injections(path):
    """The injection table a drop-in run wrote (DetectTrails(injections=...), one line per injection) as an
    INJECTION_DTYPE array; trail fields past ``ntrails`` are NaN (table indices -1)."""
    with open(path) as f:
        lines = [ln.split() for ln in f if ln.strip()]
    out = np.zeros(len(lines), INJECTION_DTYPE)
    for f in _TRAIL_F:
        out[f] = np.nan
    out["profile"] = out["lightcurve"] = -1
    for r, t in enumerate(lines):
        n = int(t[12])
        if len(t) != 13 + 8 * n or n > _T:
            raise ValueError("%s: malformed injection line %d" % (path, r + 1))
        out["run"][r], out["camcol"][r], out["filter"][r], out["field"][r], out["k"][r] = int(t[0]), int(t[1]), t[2], int(t[3]), int(t[4])
        out["base_detected"][r], out["detected"][r] = bool(int(t[5])), bool(int(t[6]))
        out["pass"][r], out["status"][r] = int(t[7]), int(t[8])
        out["rho"][r], out["theta"][r] = float(t[9]), float(t[10])
        out["recovered"][r], out["ntrails"][r] = int(t[11]), n
        if n:
            v = np.array(t[13:], dtype=object).reshape(n, 8)
            for j, fld in enumerate(_TRAIL_F):
                out[fld][r, :n] = [float(s) for s in v[:, j]]
            out["profile"][r, :n] = [int(s) for s in v[:, 6]]
            out["lightcurve"][r, :n] = [int(s) for s in v[:, 7]]
    return out


def recovery(frames, rects, injections, params_bright=None, params_dim=None, device=0, batch=64,
             theta_tol=np.deg2rad(2), rho_tol=None, tables=None):
    """Run every injection and every base without a trail; one RECOVERY_DTYPE row per injection.

    ``frames``: (n_base, H, W) un-flipped float32 bases; ``rects``: their star rectangles (lfd_submit's convention, one
    array per base) or None; ``injections``: a sequence of ``(base_index, [trail, ...])`` with at most 16 trails each;
    ``tables``: the ``(lo, hi, samples)`` tables (e.g. ``defocus_profile``) that trails' ``"profile"`` and
    ``"lightcurve"`` keys index.  The row's ``sigma`` is NaN for a tabulated profile that has none.

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
            if tables:
                h.set_trail_tables(tables)

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
        row["recovered"] = _recovered(r, ts, (H, W), hough, theta_tol, rho_tol)
    return out
