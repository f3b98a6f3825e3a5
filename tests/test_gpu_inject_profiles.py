"""Tabulated trail shapes on the device (lfd_set_trail_tables / lfd_submit_injected_shaped, k_inject): shapes of all -1
against lfd_submit_injected, tabulated profiles and light curves bit for bit against
tests/inject_shapes_ref.py::render_trails(..., tables), defocused-meteor injections against the oracle's verdicts and the
production path, recovery() with tables, and the argument checks."""
import ctypes
import math
import multiprocessing as mp
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from lfd_b200 import _lib, synth
from lfd_b200.inject import defocus_profile, recovery, trail_line
from oracle import ref_pipeline as rp
from inject_shapes_ref import footprint, render_trails
from oracle.verdicts import device_verdict, verdicts

B, NB = 64, 16
H, W = synth.FRAME_H, synth.FRAME_W
PB, PD, PR = dict(rp.DEFAULT_BRIGHT), dict(rp.DEFAULT_DIM), dict(rp.DEFAULT_REMOVESTARS)


def _gen(job):
    return synth.make_case(*job)


@pytest.fixture(scope="module")
def bases():
    """16 config-3 frames with their catalogs, filters, kinds and star rectangles."""
    from lfd_b200.removestars import star_rects
    jobs = [synth.case_for_frame(3015, 2, synth.FILTERS[i % 5], 700 + i) for i in range(NB)]
    filters = [synth.FILTERS[i % 5] for i in range(NB)]
    with mp.get_context("fork").Pool(min(os.cpu_count() or 1, NB)) as pool:
        made = pool.map(_gen, jobs, chunksize=1)
    frames = np.stack([m[0] for m in made])
    cats = [m[1] for m in made]
    rects = [star_rects(c, flt, frames[0].shape, **PR) for c, flt in zip(cats, filters)]
    return {"frames": frames, "cats": cats, "filters": filters, "kinds": [j[0] for j in jobs], "rects": rects}


def _tables():
    rng = np.random.default_rng(11)
    d4096 = np.linspace(-20.0, 20.0, 4096)
    rise = np.linspace(0.0, 1.0, 64)
    return [
        (-2.5, 7.0, rng.uniform(-0.2, 1.0, 57).astype(np.float32)),                       # 0 asymmetric, some < 0
        (-1.5, 1.5, np.array([1.0, 0.25], np.float32)),                                    # 1 n = 2
        (-20.0, 20.0, (np.cos(d4096 / 3.0) * np.exp(-np.abs(d4096) / 8)).astype(np.float32)),   # 2 n = 4096
        (-0.3, 0.4, np.array([0.5, 1.0, 0.75, 1.0, 0.6], np.float32)),                     # 3 narrower than 1 px
        (-60.0, 60.0, (0.5 + 0.5 * np.cos(np.linspace(-math.pi, math.pi, 481))).astype(np.float32)),  # 4 +-60 px
        (-5.0, 5.0, -np.exp(-0.5 * np.linspace(-5, 5, 41) ** 2).astype(np.float32)),       # 5 negative samples
        defocus_profile(6.5, 2.6, 3.5),                                                    # 6 donut
        (0.0, 1.0, np.where(rise < 0.3, (rise / 0.3) ** 2, np.exp(-(rise - 0.3) / 0.35)).astype(np.float32)),  # 7 lc
        (0.0, 1.0, np.array([0.2, 1.5], np.float32)),                                      # 8 lc, n = 2
        (-3.0, 3.0, rng.uniform(-0.5, 2.0, 4096).astype(np.float32)),                      # 9 lc, n = 4096
    ]


PROFILES, LIGHTCURVES = (0, 1, 2, 3, 4, 5, 6), (7, 8, 9)


def _t(ang_deg, cx, cy, length, peak, profile=-1, lightcurve=-1, sigma=2.0):
    a = np.deg2rad(ang_deg)
    tr = {"p0": (float(np.float32(cx - length / 2 * math.cos(a))), float(np.float32(cy - length / 2 * math.sin(a)))),
          "p1": (float(np.float32(cx + length / 2 * math.cos(a))), float(np.float32(cy + length / 2 * math.sin(a)))),
          "sigma": float(np.float32(sigma)), "peak": float(np.float32(peak))}
    if profile >= 0:
        tr["profile"] = profile
    if lightcurve >= 0:
        tr["lightcurve"] = lightcurve
    return tr


def _check_slot(got, base, ts, tables, what):
    """Bit-identical to render_trails wherever no Gaussian trail covers a pixel (the base itself outside every
    footprint); within 4 ulps per covering Gaussian trail elsewhere (expf)."""
    ref = render_trails(base.copy(), ts, tables)
    gcov = np.zeros((H, W), np.int32)
    mag = np.abs(ref).astype(np.float64)
    bound = np.zeros((H, W), np.float64)
    anyfp = np.zeros((H, W), bool)
    for tr in ts:
        fp = footprint((H, W), tr, tables)
        if fp is None:
            continue
        ya, yb, xa, xb, inside, _ = fp
        anyfp[ya:yb, xa:xb] |= inside
        pmax = 1.0 if tr.get("profile", -1) < 0 else float(np.abs(tables[tr["profile"]][2]).max())
        amax = 1.0 if tr.get("lightcurve", -1) < 0 else float(np.abs(tables[tr["lightcurve"]][2]).max())
        bound[ya:yb, xa:xb] += np.where(inside, abs(tr["peak"]) * pmax * amax, 0.0)
        if tr.get("profile", -1) < 0:
            gcov[ya:yb, xa:xb] += inside
    assert np.array_equal(got[~anyfp].view(np.uint32), base[~anyfp].view(np.uint32)), what + ": pixels outside changed"
    ex = gcov == 0
    assert np.array_equal(got[ex].view(np.uint32), ref[ex].view(np.uint32)), \
        what + ": %d pixels differ" % int((got[ex].view(np.uint32) != ref[ex].view(np.uint32)).sum())
    g = ~ex
    tol = 4 * gcov[g] * np.spacing(np.maximum(mag[g], bound[g]).astype(np.float32))
    err = np.abs(got[g].astype(np.float64) - ref[g].astype(np.float64))
    assert np.all(err <= tol), what + ": %d pixels beyond 4 ulps per Gaussian trail" % int((err > tol).sum())


@pytest.fixture(scope="module")
def handles(bases):
    hs = [_lib.Handle(H, W, max_batch=B) for _ in range(2)]
    for h in hs:
        h.set_params(PB, PD)
    hs[0].set_base(bases["frames"], bases["rects"])
    hs[0].set_trail_tables(_tables())
    yield hs
    for h in hs:
        h.close()


def test_all_minus_one_is_lfd_submit_injected(bases, handles):
    hA, _ = handles
    rng = np.random.default_rng(1)
    slots = [[_t(rng.uniform(0, 180), rng.uniform(300, 1700), rng.uniform(300, 1200), rng.uniform(300, 2000),
                 rng.uniform(0.5, 20), sigma=rng.uniform(0.8, 6))] for _ in range(24)]
    bidx = np.arange(24) % NB
    hA.submit_injected(bidx, slots)
    ref = [bytes(r) for r in hA.wait()]
    taps = [hA.stage(j, 0, "input").copy() for j in range(24)]
    # explicit -1 keys take the shaped entry point
    hA.submit_injected(bidx, [[dict(t, profile=-1, lightcurve=-1) for t in ts] for ts in slots])
    assert [bytes(r) for r in hA.wait()] == ref
    kt = hA.kernel_times()
    assert kt[-1][0] == "k_inject" and kt[-1][3] == 1
    for j in range(24):
        assert np.array_equal(hA.stage(j, 0, "input").view(np.uint32), taps[j].view(np.uint32)), j
    # shapes = NULL
    offs = np.zeros(25, np.int32)
    offs[1:] = np.arange(1, 25)
    arr = np.concatenate([_lib.Handle.trails_array(ts) for ts in slots])
    bi = np.ascontiguousarray(bidx, np.int32)
    hA._ck(hA._L.lfd_submit_injected_shaped(hA.h, 24, bi.ctypes.data_as(ctypes.c_void_p), arr.ctypes.data_as(ctypes.c_void_p),
                                            None, offs.ctypes.data_as(ctypes.c_void_p), 0))
    hA._n = 24
    assert [bytes(r) for r in hA.wait()] == ref
    for j in range(24):
        assert np.array_equal(hA.stage(j, 0, "input").view(np.uint32), taps[j].view(np.uint32)), j


def _render_slots():
    rng = np.random.default_rng(40)
    s = [
        [_t(0.0, 1000, 700, 1500, 2.0, profile=0)],                                  # asymmetric, 0 deg
        [_t(90.0, 1000, 700, 1200, 5.0, profile=1)],                                 # n = 2, 90 deg
        [_t(91.0, 600, 700, 1300, 3.0, profile=2, lightcurve=7)],                    # n = 4096, rise and fade
        [_t(89.0, 1500, 700, 1300, 3.0, profile=3)],                                 # narrower than 1 px
        [_t(45.0, 1024, 744, 1800, 1.5, profile=4)],                                 # +-60 px, 45 deg
        [_t(45.0, 1024, 744, 1800, 4.0, profile=5, lightcurve=8)],                   # negative samples, lc n = 2
        [_t(135.0, 1024, 744, 1800, 6.0, profile=6, lightcurve=9)],                  # donut, lc n = 4096
        [_t(30.0, -200, 700, 1200, 2.5, profile=4)],                                 # cut by the left edge
        [_t(80.0, 2060, 700, 900, 3.5, profile=2)],                                  # centre off the right edge
        [_t(10.0, 1024, -20, 3000, 2.0, profile=4, lightcurve=7)],                   # cut by the first row
        [_t(170.0, 1024, 1500, 3000, 2.0, profile=0)],                               # cut by the last row
        [_t(0.0, 1024, 0, 2100, 1.0, profile=6), _t(0.0, 1024, 1488, 2100, 1.0, profile=0),
         _t(90.0, 0, 744, 1600, 1.0, profile=4), _t(90.0, 2047, 744, 1600, 1.0, profile=5)],   # along the four edges
        [_t(20.0, -900, -900, 500, 40.0, profile=4)],                                # wholly off the frame
        [{"p0": (500.0, 500.0), "p1": (500.0, 500.0), "peak": 9.0, "profile": 6, "lightcurve": 7},   # zero length
         _t(60.0, 800, 800, 700, 0.2, profile=3)],
        [_t(45.0, 1024, 744, 2000, 3.0, profile=6), _t(135.0, 1024, 744, 2000, -1.5, profile=0, lightcurve=9)],
    ]
    # 16 trails in one slot, Gaussian and tabulated mixed, with and without light curves
    s.append([_t(rng.uniform(0, 180), rng.uniform(400, 1600), rng.uniform(300, 1200), rng.uniform(200, 2000),
                 rng.uniform(-3, 20), profile=(-1 if k % 3 == 0 else PROFILES[k % 7]),
                 lightcurve=(LIGHTCURVES[k % 3] if k % 2 else -1), sigma=rng.uniform(0.8, 6)) for k in range(16)])
    # Gaussian trails with light curves
    s.append([_t(33.0, 1000, 700, 1500, 12.0, lightcurve=7, sigma=3.0), _t(120.0, 900, 800, 900, 0.8, lightcurve=9, sigma=1.1)])
    s.append([_t(0.5, 1000, 400, 1900, 30.0, lightcurve=8, sigma=6.0)])
    while len(s) < 44:
        s.append([_t(rng.uniform(0, 180), rng.uniform(0, W), rng.uniform(0, H), rng.uniform(100, 2600),
                     math.exp(rng.uniform(math.log(0.3), math.log(50.0))), profile=int(rng.choice(PROFILES)),
                     lightcurve=int(rng.choice((-1,) + LIGHTCURVES))) for _ in range(int(rng.integers(1, 4)))])
    return s


def test_tabulated_rendering_matches_render_trails(bases, handles):
    hA, _ = handles
    tables = _tables()
    slots = _render_slots()
    bidx = np.arange(len(slots)) * 5 % NB
    hA.submit_injected(bidx, slots)
    hA.wait()
    for j, ts in enumerate(slots):
        _check_slot(hA.stage(j, 0, "input"), bases["frames"][bidx[j]], ts, tables, "slot %d" % j)


def _donut_grid(rng, n, tables_base):
    """Defocused meteors: r_outer 4-12 px, r_inner 0.4 r_outer, seeing FWHM 3.5 px (tables tables_base ..), any angle
    (a quarter at 0 / 90 +- 1 degrees), peak 0.3-30 log-uniform, 300-2600 px long, every third with the rise-and-fade
    light curve (table 7)."""
    out = []
    for i in range(n):
        ang = (0.0, 90.0)[i % 2] + rng.uniform(-1, 1) if i % 4 == 0 else rng.uniform(0, 180)
        out.append(_t(ang, rng.uniform(0.25 * W, 0.75 * W), rng.uniform(0.25 * H, 0.75 * H), rng.uniform(300, 2600),
                      math.exp(rng.uniform(math.log(0.3), math.log(30.0))), profile=tables_base + int(rng.integers(0, 5)),
                      lightcurve=7 if i % 3 == 0 else -1))
    return out


def test_donut_verdicts_and_production_path(bases, handles, cv2mod):
    """101 donut injections: every device verdict is the oracle's on the downloaded input frame; the same frames through
    lfd_submit on the other handle give identical result bytes at n = 64 and n = 37; lfd_run_resident repeats them."""
    hA, hB = handles
    tables = _tables() + [defocus_profile(r, 0.4 * r, 3.5) for r in (4.0, 6.0, 8.0, 10.0, 12.0)]
    hA.set_trail_tables(tables)
    rng = np.random.default_rng(101)
    grid = _donut_grid(rng, B + 37, len(_tables()))
    ndet, start = 0, 0
    for n in (B, 37):
        bidx = rng.integers(0, NB, n)
        slots = [[t] for t in grid[start:start + n]]
        start += n
        hA.submit_injected(bidx, slots)
        res = hA.wait()
        got = [device_verdict(r, (H, W)) for r in res]
        inj = [hA.stage(j, 0, "input").copy() for j in range(n)]
        for j in range(0, n, 7):
            _check_slot(inj[j], bases["frames"][bidx[j]], slots[j], tables, "donut slot %d" % j)
        hB.submit(np.stack(inj), [bases["rects"][b] for b in bidx])
        res_b = hB.wait()
        assert [bytes(r) for r in res_b] == [bytes(r) for r in res], "n = %d" % n
        ref = verdicts(inj, [bases["cats"][b] for b in bidx], [bases["filters"][b] for b in bidx], PB, PD, PR)
        bad = ["slot %d (base %d): got %s, oracle %s" % (j, bidx[j], got[j], ref[j]) for j in range(n) if got[j] != tuple(ref[j])]
        assert not bad, "\n".join(bad[:10])
        ndet += sum(1 for r in ref if r[0] is True)
    assert ndet >= 10, "grid too faint: only %d detections" % ndet
    hA.run_resident(37)
    assert [bytes(r) for r in hA.wait()] == [bytes(r) for r in res_b]
    hA.set_trail_tables(_tables())


def test_recovery_with_tables(bases, cv2mod):
    sparse = [i for i, k in enumerate(bases["kinds"]) if k == "sparse"][:8]
    assert len(sparse) >= 4
    frames = bases["frames"][sparse]
    rects = [bases["rects"][i] for i in sparse]
    tables = [defocus_profile(6.5, 2.6, 3.5), _tables()[7]]
    trail = {"p0": (100.0, 200.0), "p1": (1900.0, 1300.0), "peak": 4.0, "profile": 0}
    injections = [(b, [trail]) for b in range(len(sparse))]
    injections += [(b, [dict(trail, lightcurve=1, peak=8.0)]) for b in range(len(sparse))]
    tab = recovery(frames, rects, injections, PB, PD, batch=8, tables=tables)
    assert len(tab) == len(injections)
    assert np.all(np.isnan(tab["sigma"][:, 0])) and np.all(tab["peak"][:, 0] == [t[0]["peak"] for _, t in injections])
    h = _lib.Handle(H, W, max_batch=len(injections))
    try:
        h.set_params(PB, PD)
        h.set_base(frames, rects)
        h.set_trail_tables(tables)
        h.submit_injected([b for b, _ in injections], [ts for _, ts in injections])
        res = [bytes(r) for r in h.wait()]
        inj = [h.stage(j, 0, "input").copy() for j in range(len(injections))]
    finally:
        h.close()
    for j, (b, ts) in enumerate(injections):
        _check_slot(inj[j], frames[b], ts, tables, "recovery slot %d" % j)
    ref = verdicts(inj, [bases["cats"][sparse[b]] for b, _ in injections], [bases["filters"][sparse[b]] for b, _ in injections],
                   PB, PD, PR)
    hits = [j for j, r in enumerate(ref) if r[0] is True]
    assert hits, "the oracle detects the donut on none of the sparse bases"
    for j in hits:
        assert tab[j]["detected"] and tab[j]["recovered"] == 0, (j, tab[j]["rho"], tab[j]["theta"], trail_line(trail, (H, W)))
    # recovery's verdicts are those of the same frames on this handle
    assert [bool(r[0]) for r in (np.frombuffer(x, np.dtype(_lib.Result), count=1)[0] for x in res)] == list(tab["detected"])


def _set_raw(h, samples, tab):
    s = np.ascontiguousarray(samples, np.float32)
    t = np.ascontiguousarray(np.array(tab, _lib.TABLE_DTYPE).reshape(-1))
    return h._L.lfd_set_trail_tables(h.h, s.ctypes.data_as(ctypes.c_void_p), len(s), t.ctypes.data_as(ctypes.c_void_p), len(t))


def test_argument_checks_launch_nothing():
    h = _lib.Handle(H, W, max_batch=4)
    rng = np.random.default_rng(3)
    frames = rng.standard_normal((2, H, W), dtype=np.float32) * np.float32(0.025)
    try:
        h.set_params(PB, PD)

        def code(fn, *a, **k):
            with pytest.raises(_lib.LfdError) as e:
                fn(*a, **k)
            return e.value.code

        l0 = h.kernel_launches()
        h.set_base(frames)
        ok = _t(30.0, 1000, 700, 1000, 3.0)
        assert code(h.submit_injected, [0], [[dict(ok, profile=0)]]) == _lib.LFD_E_STATE        # no pool yet
        assert code(h.submit_injected, [0], [[dict(ok, lightcurve=0)]]) == _lib.LFD_E_STATE
        smp = np.linspace(0, 1, 100, dtype=np.float32)
        E = _lib.LFD_E_ARG
        assert _set_raw(h, smp, [(0, 1, -1.0, 1.0)]) == E                  # n = 1
        assert _set_raw(h, np.zeros(5000, np.float32), [(0, 4097, -1.0, 1.0)]) == E             # n = 4097
        assert _set_raw(h, smp, [(0, 101, -1.0, 1.0)]) == E                # past the samples
        assert _set_raw(h, smp, [(-1, 10, -1.0, 1.0)]) == E                # before the samples
        assert _set_raw(h, smp, [(95, 10, -1.0, 1.0)]) == E
        bad = smp.copy()
        bad[50] = np.nan
        assert _set_raw(h, bad, [(0, 10, -1.0, 1.0)]) == E                 # a non-finite sample
        bad[50] = np.inf
        assert _set_raw(h, bad, [(0, 10, -1.0, 1.0)]) == E
        assert _set_raw(h, smp, [(0, 10, -np.inf, 1.0)]) == E              # lo / hi not finite
        assert _set_raw(h, smp, [(0, 10, -1.0, np.nan)]) == E
        assert _set_raw(h, smp, [(0, 10, 1.0, 1.0)]) == E                  # lo >= hi
        assert _set_raw(h, smp, [(0, 10, 2.0, 1.0)]) == E
        assert _set_raw(h, smp, [(0, 10, -1024.5, 1.0)]) == E              # max(|lo|, |hi|) > 1024
        assert _set_raw(h, smp, [(0, 10, 0.0, 1025.0)]) == E
        assert _set_raw(h, smp, [(0, 10, -1.0, 1.0)] * 4097) == E          # more than 4096 tables
        assert _set_raw(h, smp, []) == E
        assert _set_raw(h, smp, [(0, 10, -1024.0, 1024.0)] * 4096) == _lib.LFD_OK   # the limits themselves
        assert _set_raw(h, np.zeros(4096, np.float32), [(0, 4096, -1.0, 1.0)]) == _lib.LFD_OK
        h.set_trail_tables([(-3.0, 3.0, np.ones(13)), (0.0, 1.0, np.ones(4))])
        for shape in ({"profile": 2}, {"lightcurve": 2}, {"profile": -2}, {"lightcurve": -7}, {"profile": 1 << 20}):
            assert code(h.submit_injected, [0, 1], [[ok], [dict(ok, **shape)]]) == E, shape
        for key, v in (("p0", (math.nan, 1.0)), ("p1", (1.0, math.inf)), ("peak", math.inf)):
            assert code(h.submit_injected, [0], [[dict(ok, profile=0, **{key: v})]]) == E, key
        assert code(h.submit_injected, [0], [[dict(ok, sigma=0.0, lightcurve=1)]]) == E       # Gaussian: sigma checked
        assert h.kernel_launches() == l0, "a rejected call launched a kernel"
        # set_trail_tables while a batch is pending
        h.submit_injected([0], [[dict(ok, profile=0, sigma=math.nan)]])              # tabulated: sigma not checked
        assert code(h.set_trail_tables, [(-3.0, 3.0, np.ones(13))]) == _lib.LFD_E_STATE
        h.wait()
        tap = h.stage(0, 0, "input")
        ref = render_trails(frames[0].copy(), [dict(ok, profile=0)], [(-3.0, 3.0, np.ones(13))])
        assert np.array_equal(tap.view(np.uint32), ref.view(np.uint32))
    finally:
        h.close()


def test_replacing_the_pool_takes_effect(bases, handles):
    hA, _ = handles
    t1 = [(-4.0, 4.0, np.linspace(0.0, 1.0, 17).astype(np.float32)), (0.0, 1.0, np.array([1.0, 0.1], np.float32))]
    t2 = [(-9.0, 2.0, np.linspace(1.0, -0.5, 300).astype(np.float32)), (0.0, 1.0, np.array([0.1, 2.0, 0.3], np.float32))]
    slots = [[_t(25.0, 1000, 700, 1400, 5.0, profile=0, lightcurve=1)], [_t(100.0, 700, 700, 900, 2.0, profile=0)]]
    taps = []
    try:
        for tabs in (t1, t2):
            hA.set_trail_tables(tabs)
            hA.submit_injected([3, 4], slots)
            hA.wait()
            taps.append([hA.stage(j, 0, "input").copy() for j in range(2)])
            for j in range(2):
                _check_slot(taps[-1][j], bases["frames"][3 + j], slots[j], tabs, "pool %d slot %d" % (len(taps), j))
        assert not np.array_equal(taps[0][0], taps[1][0])
    finally:
        hA.set_trail_tables(_tables())
