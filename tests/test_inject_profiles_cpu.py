"""Tabulated trail shapes on the host: tests/inject_shapes_ref.py::render_trails with tables (cross-section profiles and light
curves, include/lfd_b200.h lfd_table) against the Gaussian it generalises, and lfd_b200.inject.defocus_profile."""
import math

import numpy as np
import pytest

from lfd_b200.inject import _defocus_samples, defocus_profile
from inject_shapes_ref import footprint, render_trails
from oracle import inject_ref
from oracle.inject_ref import trail_params

H, W = 160, 200


def _base(seed=1):
    return np.random.default_rng(seed).standard_normal((H, W)).astype(np.float32) * np.float32(0.05)


TRAILS = [
    {"p0": (10.5, 20.25), "p1": (180.0, 140.0), "sigma": 1.7, "peak": 3.0},
    {"p0": (100.0, -5.0), "p1": (101.0, 170.0), "sigma": 0.8, "peak": 0.7},          # about 90 degrees, cut by two edges
    {"p0": (-20.0, 80.0), "p1": (220.0, 80.0), "sigma": 4.0, "peak": -1.5},          # 0 degrees, negative
]


def test_without_shapes_it_is_the_oracle():
    a = inject_ref.render_trails(_base(), TRAILS)
    b = render_trails(_base(), TRAILS)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    for tr in TRAILS:
        fa, fb = inject_ref.footprint((H, W), tr), footprint((H, W), tr)
        assert fa[:4] == fb[:4] and np.array_equal(fa[4], fb[4])
        assert np.array_equal(fa[5].view(np.uint32), fb[5].view(np.uint32))


@pytest.mark.parametrize("tr", TRAILS)
def test_all_ones_table_adds_peak_over_the_gaussian_footprint(tr):
    pad = float(trail_params(tr)[7])
    tables = [(-pad, pad, np.ones(7, np.float32))]
    g = footprint((H, W), tr)
    t = footprint((H, W), dict(tr, profile=0), tables)
    assert g[:4] == t[:4]
    assert np.array_equal(g[4], t[4])
    base = _base()
    got = render_trails(base.copy(), [dict(tr, profile=0)], tables)
    exp = base.copy()
    ya, yb, xa, xb, ins = g[:5]
    exp[ya:yb, xa:xb][ins] += np.float32(tr["peak"])
    assert np.array_equal(got.view(np.uint32), exp.view(np.uint32))


def test_tabulated_profile_ignores_sigma():
    tables = [(-3.0, 5.0, np.array([0.0, 8.0], np.float32))]       # asymmetric, n = 2: P = d + 3
    tr = dict(TRAILS[0], profile=0)
    a = render_trails(_base(), [tr], tables)
    b = render_trails(_base(), [{k: v for k, v in tr.items() if k != "sigma"}], tables)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    ya, yb, xa, xb, ins, add = footprint((H, W), tr, tables)
    x0, y0, ux, uy = (float(v) for v in trail_params(dict(tr, sigma=1.0))[:4])
    yy, xx = np.mgrid[ya:yb, xa:xb]
    d = -(xx - x0) * uy + (yy - y0) * ux
    assert d[ins].min() >= -3.0 - 1e-4 and d[ins].max() <= 5.0 + 1e-4
    assert np.allclose(add[ins], float(tr["peak"]) * (d[ins] + 3.0), atol=1e-4)


@pytest.mark.parametrize("profile", [-1, 0])
def test_constant_light_curve_is_no_light_curve(profile):
    tables = [(-6.0, 4.0, np.linspace(0.2, 1.0, 33, dtype=np.float32)), (0.0, 1.0, np.ones(64, np.float32))]
    trs = [dict(t, profile=profile) for t in TRAILS]
    a = render_trails(_base(), trs, tables)
    b = render_trails(_base(), [dict(t, lightcurve=1) for t in trs], tables)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


def test_light_curve_spans_the_segment():
    tr = {"p0": (20.0, 50.0), "p1": (180.0, 50.0), "peak": 2.0, "profile": 0, "lightcurve": 1}
    tables = [(-2.0, 2.0, np.ones(5, np.float32)), (0.0, 1.0, np.array([0.0, 1.0], np.float32))]
    img = render_trails(np.zeros((H, W), np.float32), [tr], tables)
    row = img[50, 20:181]
    assert np.allclose(row, 2.0 * np.arange(161) / 160.0, atol=1e-5)     # rises linearly from p0 to p1
    assert img[50, 19] == 0 and img[50, 181] == 0


@pytest.mark.parametrize("tr", TRAILS)
def test_sampled_gaussian_matches_the_gaussian(tr):
    sigma, pad = float(trail_params(tr)[5]), float(trail_params(tr)[7])
    d = np.linspace(-pad, pad, int(round(2 * pad * 64)) + 1)
    tables = [(-pad, pad, np.exp(-0.5 * (d / sigma) ** 2).astype(np.float32))]
    base = _base()
    g = render_trails(base.copy(), [tr], tables)
    t = render_trails(base.copy(), [dict(tr, profile=0)], tables)
    # linear interpolation error (1/64)^2 / 8 * max|f''| with max|f''| = 1 / sigma^2, plus float32 rounding
    tol = abs(tr["peak"]) * ((1 / 64) ** 2 / 8 / sigma ** 2 + 1e-6) + 4 * np.spacing(np.abs(g))
    assert np.all(np.abs(t.astype(np.float64) - g) <= tol)


def test_defocus_profile_shape():
    for args in ((6.5, 2.6, 0.0), (6.5, 2.6, 3.5), (12.0, 4.8, 3.5), (4.0, 0.0, 0.0), (0.0, 0.0, 3.5)):
        lo, hi, p = defocus_profile(*args)
        assert p.dtype == np.float32 and len(p) == int(round((hi - lo) / 0.25)) + 1
        assert lo == -hi and hi >= args[0] + 4 * args[2] / 2.3548 - 1e-9 and (hi / 0.25) == int(hi / 0.25)
        assert np.array_equal(p, p[::-1]), args
        assert p.max() == 1.0
    # 2.5 m at 100 km, 0.396 arcsec / px: r_outer = 6.5 px; the seeing fills the central dip only partly
    lo, hi, p = defocus_profile(6.5, 2.6, 3.5)
    c = len(p) // 2
    assert p[c] < p.max() and lo == -12.5


@pytest.mark.parametrize("ro, ri", [(6.5, 2.5), (12.0, 4.75), (4.0, 0.0), (9.0, 9.0 * 0.4)])
def test_defocus_profile_centre_over_maximum(ro, ri):
    step = 0.25 if ri / 0.25 == int(ri / 0.25) else 0.05
    lo, hi, p = defocus_profile(ro, ri, 0.0, step)
    exp = (ro - ri) / math.sqrt(ro * ro - ri * ri)
    assert abs(float(p[len(p) // 2]) - exp) <= 1e-6
    d = lo + step * np.arange(len(p))
    assert np.all(np.abs(np.abs(d[p == p.max()]) - ri) < 1e-6)


@pytest.mark.parametrize("ro, ri", [(6.5, 2.6), (12.0, 4.8), (4.0, 1.6), (8.0, 0.0)])
def test_defocus_profile_integral(ro, ri):
    exp = math.pi * (ro * ro - ri * ri) / 2
    step = 1 / 32
    d, a = _defocus_samples(ro, ri, 0.0, step)
    assert abs(a.sum() * step / exp - 1) <= 1e-3
    for fw in (1.0, 3.5, 8.0):
        for st in (step, 0.25):
            d, a = _defocus_samples(ro, ri, fw, st)
            assert abs(a.sum() * st / exp - 1) <= 1e-3, (fw, st)


@pytest.mark.parametrize("args", [(0.0, 0.0, 0.0), (-1.0, 0.0, 0.0), (5.0, 6.0, 1.0), (5.0, -1.0, 0.0),
                                  (5.0, 1.0, -1.0), (5.0, 1.0, 1.0, 0.0), (math.nan, 0.0, 1.0), (600.0, 0.0, 0.0)])
def test_defocus_profile_rejects(args):
    with pytest.raises(ValueError):
        defocus_profile(*args)
