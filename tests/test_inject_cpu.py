"""Injection without a GPU: the NumPy reference of the injected trail (oracle/inject_ref.py) against synth's renderer,
the line geometry of lfd_b200/inject.py::trail_line, and the matching rule on the oracle's own detections."""
import math
import multiprocessing as mp
import os

import numpy as np
import pytest

from lfd_b200 import synth
from lfd_b200.inject import _first_match, trail_line
from oracle.inject_ref import render_trails


def _f32(v):
    return float(np.float32(v))


def _random_trails(rng, n, h, w):
    out = []
    for i in range(n):
        p0 = (_f32(rng.uniform(-150, w + 150)), _f32(rng.uniform(-150, h + 150)))
        p1 = (_f32(rng.uniform(-150, w + 150)), _f32(rng.uniform(-150, h + 150)))
        if i % 5 == 0:
            p1 = (_f32(p0[0] + rng.uniform(-300, 300)), p0[1])           # horizontal
        elif i % 5 == 1:
            p1 = (p0[0], _f32(p0[1] + rng.uniform(-300, 300)))           # vertical
        out.append({"p0": p0, "p1": p1, "sigma": _f32(rng.uniform(0.8, 6.4)), "peak": _f32(rng.uniform(-3, 50))})
    return out


def test_render_trails_matches_synth_where_both_add():
    rng = np.random.default_rng(20261020)
    h, w = 300, 400
    both_total = 0
    for tr in _random_trails(rng, 40, h, w):
        base = rng.standard_normal((h, w), dtype=np.float32)
        a = base.copy()
        synth._add_trail(a, tr["p0"], tr["p1"], tr["sigma"], tr["peak"])
        b = render_trails(base.copy(), [tr])
        add_a = a.view(np.uint32) != base.view(np.uint32)
        add_b = b.view(np.uint32) != base.view(np.uint32)
        both = add_a & add_b
        assert np.array_equal(a[both].view(np.uint32), b[both].view(np.uint32)), tr
        # where only render_trails adds, _add_trail added an exact zero (its tails underflow or pass through +0)
        x0, y0 = tr["p0"]
        x1, y1 = tr["p1"]
        pad = int(np.ceil(5 * tr["sigma"])) + 1
        box = np.zeros((h, w), bool)
        ya, yb = max(int(min(y0, y1)) - pad, 0), min(int(max(y0, y1)) + pad + 1, h)
        xa, xb = max(int(min(x0, x1)) - pad, 0), min(int(max(x0, x1)) + pad + 1, w)
        box[ya:yb, xa:xb] = True
        assert not np.any(add_b & ~box), "render_trails added flux outside _add_trail's bounding box"
        both_total += int(both.sum())
    assert both_total > 100000


def test_render_trails_zero_length_and_order():
    img = np.zeros((64, 64), np.float32)
    render_trails(img, [{"p0": (10.0, 10.0), "p1": (10.0, 10.0), "sigma": 2.0, "peak": 5.0}])
    assert not img.any()
    t1 = {"p0": (0.0, 30.0), "p1": (63.0, 30.0), "sigma": 1.5, "peak": 7.0}
    t2 = {"p0": (30.0, 0.0), "p1": (30.0, 63.0), "sigma": 2.5, "peak": -0.3}
    a = render_trails(np.full((64, 64), 0.1, np.float32), [t1, t2])
    b = render_trails(render_trails(np.full((64, 64), 0.1, np.float32), [t1]), [t2])
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    assert a[30, 10] == np.float32(0.1) + np.float32(7.0)
    # the footprint stops at |d| = ceil(5 sigma) + 1 = 9 px for sigma 1.5
    assert a[30 + 9, 10] != np.float32(0.1) and a[30 + 10, 10] == np.float32(0.1)


def _on_line(rho, theta, x, yf):
    return x * math.cos(theta) + yf * math.sin(theta) - rho


@pytest.mark.parametrize("p0,p1,exp", [
    ((100.0, 200.0), (900.0, 200.0), (1488 - 200.0, math.pi / 2)),      # horizontal
    ((900.0, 200.0), (100.0, 200.0), (1488 - 200.0, math.pi / 2)),
    ((300.0, 50.0), (300.0, 1400.0), (300.0, 0.0)),                    # vertical
    ((300.0, 1400.0), (300.0, 50.0), (300.0, 0.0)),
    ((0.0, 1488.0), (1000.0, 488.0), (0.0, 3 * math.pi / 4)),           # y' = x in the flipped frame
    ((0.0, 0.0), (1000.0, 1000.0), (1488 / math.sqrt(2), math.pi / 4)),  # y' = 1488 - x
])
def test_trail_line_known_lines(p0, p1, exp):
    rho, theta = trail_line({"p0": p0, "p1": p1}, (1489, 2048))
    assert 0 <= theta < math.pi
    assert rho == pytest.approx(exp[0], abs=1e-9) and theta == pytest.approx(exp[1], abs=1e-12)


def test_trail_line_both_sides_of_the_wrap():
    H = 1489
    for deg in (-1.0, -0.25, 0.25, 1.0):              # near-vertical segments: theta just above 0 or just below pi
        a = np.deg2rad(90 + deg)
        p0 = (1000.0 - 600 * math.cos(a), 700.0 - 600 * math.sin(a))
        p1 = (1000.0 + 600 * math.cos(a), 700.0 + 600 * math.sin(a))
        rho, theta = trail_line({"p0": p0, "p1": p1}, (H, 2048))
        assert 0 <= theta < math.pi
        assert min(theta, math.pi - theta) == pytest.approx(abs(np.deg2rad(deg)), abs=1e-12)
        for x, y in (p0, p1):
            assert abs(_on_line(rho, theta, x, H - 1 - y)) < 1e-9
        # the same line written from the other side of the wrap has the opposite rho
        # a detection 1.5 degrees away on the other side of the wrap, so with the opposite rho
        near = theta - math.pi + np.deg2rad(1.5) if theta > math.pi / 2 else theta + math.pi - np.deg2rad(1.5)
        assert 0 <= near < math.pi
        assert _first_match(-rho, near, [(rho, theta)], np.deg2rad(2), 20.0) == 0
        assert _first_match(rho, near, [(rho, theta)], np.deg2rad(2), 20.0) == -1
        assert _first_match(-rho, near, [(rho, theta)], np.deg2rad(1), 20.0) == -1
        assert _first_match(rho + 25.0, theta, [(rho, theta)], np.deg2rad(2), 20.0) == -1
    assert math.isnan(trail_line({"p0": (5.0, 5.0), "p1": (5.0, 5.0)}, (H, 2048))[0])


def _case_trail(kind, seed):
    """The trail synth.make_case draws for ``kind`` (its first rng draws, replayed)."""
    if kind == "trail":
        return {"p0": (100, 200), "p1": (1900, 1300), "sigma": 3.0, "peak": 3.0}
    rng = np.random.default_rng(seed ^ 0xABCDEF)
    rng.integers(100, 500)
    return synth._random_trail(rng)


def _oracle_line(job):
    import cv2
    cv2.setNumThreads(1)
    from oracle import ref_pipeline as rp
    kind, seed = job
    img, cat = synth.make_case(kind, seed)
    taps = {}
    det, p, _ = rp.process_frame(img, cat, "r", taps=taps)
    if not det:
        return None
    return p, tuple(float(v) for v in taps[("bright", "dim")[p]]["lines_equ"][0][0])


def test_oracle_detections_match_their_trails(cv2mod):
    from oracle import ref_pipeline as rp
    jobs = [("trail", 500 + i) for i in range(4)] + [("trail_var", 600 + i) for i in range(8)]
    with mp.get_context("fork").Pool(min(os.cpu_count() or 1, len(jobs))) as pool:
        got = pool.map(_oracle_line, jobs, chunksize=1)
    ndet = 0
    for job, g in zip(jobs, got):
        if g is None:
            continue
        ndet += 1
        p, (rho, theta) = g
        hm = (rp.DEFAULT_BRIGHT, rp.DEFAULT_DIM)[p]["houghMethod"]
        tl = trail_line(_case_trail(*job), (synth.FRAME_H, synth.FRAME_W))
        assert _first_match(rho, theta, [tl], np.deg2rad(2), hm) == 0, (job, (rho, theta), tl)
    assert ndet >= 6, "only %d of %d trail frames detected" % (ndet, len(jobs))
