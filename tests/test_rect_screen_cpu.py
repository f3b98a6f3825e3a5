"""The aspect screen of k_rects_screen (lfd_b200/csrc/k_rects.cuh), restated in NumPy and checked against cv2.minAreaRect.

For a point set P whose minimum-area rectangle has sides length >= width: length <= D (the diagonal of P's bounding box),
width * D >= area(hull(P)) >= A (the area of the polygon through P's row extremes), so length / width <= D^2 / A.  The
screen rejects a contour when D^2 * (1 + 1e-4) < lwTresh * A; no rejected contour may have a rectangle that passes
fit_minAreaRect's filter (processfield.py:256-257), at any minAreaRectMinLen."""
import numpy as np
import pytest

from oracle import ref_pipeline as rp

MARGIN = 1e-4                     # SCREEN_MARGIN
LW = (0.5, 1.0, 2.0, 5.0, 20.0)
MINLEN = (0.0, 1.0, 3.0)


def screen_terms(pts):
    """(D^2, 2A) of a point set (x, y int): the squared bounding-box diagonal and twice the area of the polygon through
    the row extremes, summed over consecutive non-empty rows like the kernel."""
    pts = np.asarray(pts, np.int64).reshape(-1, 2)
    xs, ys = pts[:, 0], pts[:, 1]
    order = np.lexsort((xs, ys))
    ys_s, xs_s = ys[order], xs[order]
    rows = np.unique(ys_s)
    rmin = xs_s[np.searchsorted(ys_s, rows, "left")]
    rmax = xs_s[np.searchsorted(ys_s, rows, "right") - 1]
    w = rmax - rmin
    a2 = int(((rows[1:] - rows[:-1]) * (w[1:] + w[:-1])).sum())
    bw, bh = int(xs.max() - xs.min()), int(ys.max() - ys.min())
    return bw * bw + bh * bh, a2


def screen_rejects(pts, lwTresh):
    d2, a2 = screen_terms(pts)
    return float(d2) * (1.0 + MARGIN) < lwTresh * (0.5 * float(a2))


def passes(rect, minLen, lwTresh):
    """processfield.py:256-257 on a cv2.minAreaRect result (float32 sides, compared in double like emit_rect)."""
    w, h = rect[1]
    length, width = (w, h) if w > h else (h, w)
    return length > minLen and width > minLen and length / width > lwTresh


def _unsound(cv2, point_sets):
    """Every (set index, lwTresh, minLen) where the screen rejects a set whose rectangle passes."""
    bad = []
    for i, pts in enumerate(point_sets):
        rect = cv2.minAreaRect(np.asarray(pts, np.int32).reshape(-1, 1, 2))
        for lw in LW:
            if screen_rejects(pts, lw):
                bad += [(i, lw, ml) for ml in MINLEN if passes(rect, ml, lw)]
    return bad


def _random_sets(cv2):
    rng = np.random.default_rng(20261022)
    sets = []
    for deg in np.arange(0.0, 180.0, 2.5):                  # thin lines at every angle, 1 and 2 px wide
        for L in (3, 12, 60):
            for th in (1, 2):
                img = np.zeros((160, 160), np.uint8)
                t = np.radians(deg)
                p0 = (80 - int(round(L * np.cos(t))), 80 - int(round(L * np.sin(t))))
                p1 = (80 + int(round(L * np.cos(t))), 80 + int(round(L * np.sin(t))))
                cv2.line(img, p0, p1, 255, th)
                sets.append(np.argwhere(img)[:, ::-1])
    for r in (1, 2, 3, 5, 8, 20, 45):                       # rings, circles, ellipses
        img = np.zeros((128, 128), np.uint8)
        cv2.circle(img, (64, 64), r, 255, 1)
        sets.append(np.argwhere(img)[:, ::-1])
        img[:] = 0
        cv2.ellipse(img, (64, 64), (r + 10, max(1, r // 3)), float(rng.integers(0, 180)), 0, 360, 255, 1)
        sets.append(np.argwhere(img)[:, ::-1])
    for r in (2, 6, 15):                                    # filled discs and tilted filled rectangles
        img = np.zeros((64, 64), np.uint8)
        cv2.circle(img, (32, 32), r, 255, -1)
        sets.append(np.argwhere(img)[:, ::-1])
        for deg in (0, 20, 45):
            img[:] = 0
            box = cv2.boxPoints(((32, 32), (2 * r + 1, r + 1), deg))
            cv2.fillPoly(img, [np.rint(box).astype(np.int32)], 255)
            sets.append(np.argwhere(img)[:, ::-1])
    for n in (1, 2, 5, 40):                                 # single rows, single columns
        sets.append(np.stack([np.arange(n) + 7, np.full(n, 3)], 1))
        sets.append(np.stack([np.full(n, 3), np.arange(n) + 7], 1))
    for x in range(3):                                      # single pixels, pairs
        sets.append(np.array([[x, 5]]))
        sets.append(np.array([[x, 5], [x + 1, 6]]))
    for _ in range(300):                                    # random clouds, some thin, some sparse
        n = int(rng.integers(2, 60))
        sx, sy = rng.uniform(0.3, 30.0, 2)
        pts = np.stack([rng.normal(50, sx, n), rng.normal(50, sy, n)], 1)
        sets.append(np.unique(np.clip(np.rint(pts), 0, 100).astype(np.int64), axis=0))
    return sets


def test_bound_terms_exact_on_shapes():
    """D^2 and 2A of hand-made sets: a filled square's row polygon is the square itself, a diagonal line encloses
    nothing, a pixel has no extent."""
    sq = np.array([[x, y] for x in range(5) for y in range(5)])
    assert screen_terms(sq) == (32, 32)
    assert screen_terms(np.array([[i, i] for i in range(9)])) == (128, 0)
    assert screen_terms(np.array([[3, 4]])) == (0, 0)
    ring = np.array([[0, 0], [4, 0], [0, 2], [4, 2], [0, 4], [4, 4]])        # rowmin / rowmax only: still the square
    assert screen_terms(ring) == (32, 32)
    gap = np.array([[0, 0], [2, 0], [0, 3], [2, 3]])                         # empty rows: spanned by one trapezoid
    assert screen_terms(gap) == (13, 12)
    assert not any(screen_rejects(sq, lw) for lw in (0.5, 1.0, float("nan")))
    assert screen_rejects(sq, 2.0 + 1e-6) is False and screen_rejects(sq, 2.0 * (1 + 2e-4)) is True


def test_screen_sound_on_random_point_sets(cv2mod):
    """Thin lines at every angle, rings, ellipses, single rows and pixels, random clouds; lwTresh in {0.5, 1, 2, 5, 20},
    minAreaRectMinLen in {0, 1, 3}: no rejected set has a passing rectangle."""
    sets = _random_sets(cv2mod)
    bad = _unsound(cv2mod, sets)
    assert not bad, bad[:10]
    rej = {lw: sum(screen_rejects(p, lw) for p in sets) for lw in LW}
    print("random sets: %d, rejected per lwTresh %s" % (len(sets), rej))
    # A <= bw * bh <= D^2 / 2: no rejection at lwTresh <= 2
    assert rej[0.5] == rej[1.0] == rej[2.0] == 0 and rej[5.0] > 0


def _pool_contours(cv2, nframes, params):
    """cv2's contours (RETR_LIST, CHAIN_APPROX_NONE) of both passes of the first nframes frames of bench.py's pool."""
    import bench
    from lfd_b200 import synth
    frames, cats, _rects, _kinds = bench.make_pool(nframes, 0)
    pb, pd = params
    out = []
    for i, (img, cat) in enumerate(zip(frames, cats)):
        img = img.copy()
        rp.blot(img, rp.star_rects(cat, synth.FILTERS[i % 5], **rp.DEFAULT_REMOVESTARS))
        work = cv2.flip(img, 0)
        for pp, fn in ((pb, rp.bright_pass), (pd, rp.dim_pass)):
            taps = {}
            fn(work, taps=taps, **pp)
            out.append((pp, [c.reshape(-1, 2) for c in taps["contours"]], taps["rects"]))
    return out


@pytest.mark.parametrize("config", ["config3", "config4"])
def test_screen_sound_on_pool_contours(cv2mod, config):
    """Both passes of 8 frames of the config-3 pool at the config-3 (default) or config-4 (15 x 15 dilation in the dim
    pass) parameters: no contour the screen rejects at the pass's lwTresh has a passing rectangle; at the defaults the
    screen rejects more than 90 % of them."""
    pb, pd = dict(rp.DEFAULT_BRIGHT), dict(rp.DEFAULT_DIM)
    if config == "config4":
        pd["dilateKernel"] = np.ones((15, 15), np.uint8)
    total = rejected = kept = 0
    bad = []
    for pp, contours, rects in _pool_contours(cv2mod, 8, (pb, pd)):
        for pts, rect in zip(contours, rects):
            total += 1
            ok = passes(rect, pp["minAreaRectMinLen"], pp["lwTresh"])
            kept += ok
            if screen_rejects(pts, pp["lwTresh"]):
                rejected += 1
                if ok:
                    bad.append((rect, len(pts)))
        bad += [("lw", b) for b in _unsound(cv2mod, contours[:400])]
    print("%s: %d contours, %d pass, screen rejects %d (%.1f %%)" % (config, total, kept, rejected, 100.0 * rejected / total))
    assert not bad, bad[:10]
    assert total > 5000
    if config == "config3":
        assert rejected > 0.9 * total
