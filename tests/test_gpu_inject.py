"""On-device trail injection (lfd_set_base / lfd_submit_injected, k_inject) and the recovery table of
lfd_b200/inject.py: the injected frames against oracle/inject_ref.py::render_trails, every verdict against the oracle
on the frame the device read, the production path on the same frames, and the argument checks."""
import math
import multiprocessing as mp
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from lfd_b200 import _lib, synth
from lfd_b200.inject import recovery, trail_line
from oracle import ref_pipeline as rp
from oracle.inject_ref import footprint, render_trails
from oracle.verdicts import device_verdict, verdicts

B = 64
H, W = synth.FRAME_H, synth.FRAME_W
PB, PD, PR = dict(rp.DEFAULT_BRIGHT), dict(rp.DEFAULT_DIM), dict(rp.DEFAULT_REMOVESTARS)


def _gen(job):
    return synth.make_case(*job)


@pytest.fixture(scope="module")
def bases():
    """64 config-3 frames (sparse and dense mix) with their catalogs, filters, kinds and star rectangles."""
    from lfd_b200.removestars import star_rects
    jobs, filters = [], []
    for i in range(B):
        jobs.append(synth.case_for_frame(2888, 5, synth.FILTERS[i % 5], 400 + i))
        filters.append(synth.FILTERS[i % 5])
    with mp.get_context("fork").Pool(min(os.cpu_count() or 1, 32)) as pool:
        made = pool.map(_gen, jobs, chunksize=2)
    frames = np.stack([m[0] for m in made])
    cats = [m[1] for m in made]
    rects = [star_rects(c, flt, frames[0].shape, **PR) for c, flt in zip(cats, filters)]
    return {"frames": frames, "cats": cats, "filters": filters, "kinds": [j[0] for j in jobs], "rects": rects}


@pytest.fixture(scope="module")
def handles(bases):
    hs = [_lib.Handle(H, W, max_batch=B) for _ in range(2)]
    for h in hs:
        h.set_params(PB, PD)
    hs[0].set_base(bases["frames"], bases["rects"])
    yield hs
    for h in hs:
        h.close()


def _trail(ang_deg, cx, cy, length, sigma, peak):
    a = np.deg2rad(ang_deg)
    return {"p0": (float(np.float32(cx - length / 2 * math.cos(a))), float(np.float32(cy - length / 2 * math.sin(a)))),
            "p1": (float(np.float32(cx + length / 2 * math.cos(a))), float(np.float32(cy + length / 2 * math.sin(a)))),
            "sigma": float(np.float32(sigma)), "peak": float(np.float32(peak))}


def _random_grid(rng, n):
    """Trails like the config-3 mix: any angle (a quarter at 0 / 90 degrees +- 1), FWHM 2-15 px, peak 0.3-50
    log-uniform, 300-2600 px long, centred in the middle half of the frame."""
    out = []
    for i in range(n):
        ang = (0.0, 90.0)[i % 2] + rng.uniform(-1, 1) if i % 4 == 0 else rng.uniform(0, 180)
        out.append(_trail(ang, rng.uniform(0.25 * W, 0.75 * W), rng.uniform(0.25 * H, 0.75 * H), rng.uniform(300, 2600),
                          rng.uniform(2.0, 15.0) / 2.3548, math.exp(rng.uniform(math.log(0.3), math.log(50.0)))))
    return out


def test_no_trails_is_the_plain_submit(bases, handles):
    hA, hB = handles
    hA.submit_injected(np.arange(B))
    ra = [bytes(r) for r in hA.wait()]
    kt = hA.kernel_times()
    assert kt[-1][0] == "k_inject" and kt[-1][2] > 0 and kt[-1][3] == 1
    for j in range(B):
        assert np.array_equal(hA.stage(j, 0, "input").view(np.uint32), bases["frames"][j].view(np.uint32)), j
    hB.submit(bases["frames"], bases["rects"])
    rb = [bytes(r) for r in hB.wait()]
    assert all(ms == 0.0 for _n, ms in hB.timings()[2:]), "the plain submit did not take the CUDA-graph path"
    assert ra == rb
    assert hB.kernel_times() == [], "k_inject reported after a plain submit"
    # the input tap of a big-endian run is swapped back to native order
    hB.submit(bases["frames"][:3], bases["rects"][:3])
    r3 = [bytes(r) for r in hB.wait()]
    hB.submit(bases["frames"][:3].byteswap(), bases["rects"][:3], flags=_lib.INPUT_BIGENDIAN)
    assert [bytes(r) for r in hB.wait()] == r3
    for j in range(3):
        assert np.array_equal(hB.stage(j, 1, "input").view(np.uint32), bases["frames"][j].view(np.uint32))


RENDER_SLOTS = [
    [_trail(0.0, 1000, 700, 1500, 0.8, 0.05)],
    [_trail(90.0, 1000, 700, 1200, 6.4, 50.0)],
    [_trail(1.0, 900, 300, 1800, 2.0, 3.0), _trail(-1.0, 900, 1200, 1800, 3.0, 0.5)],
    [_trail(91.0, 400, 700, 1400, 1.3, 8.0), _trail(89.0, 1600, 700, 1400, 4.4, 1.0)],
    [_trail(45.0, 1024, 744, 2000, 3.0, 3.0)],
    [_trail(45.0, 1024, 744, 2000, 3.0, 3.0), _trail(135.0, 1024, 744, 2000, 2.0, -1.5)],   # crossing, one negative
    [_trail(30.0, -200, 700, 1200, 2.5, 5.0)],                       # partly off the left edge
    [_trail(10.0, 1024, -20, 3000, 5.0, 2.0)],                       # straddles the first row
    [_trail(80.0, 2060, 700, 900, 3.5, 12.0)],                       # centre off the right edge, tails inside
    [_trail(20.0, -900, -900, 500, 2.0, 40.0)],                      # wholly off the frame
    [{"p0": (500.0, 500.0), "p1": (500.0, 500.0), "sigma": 3.0, "peak": 9.0},   # zero length
     _trail(60.0, 800, 800, 700, 1.0, 0.2)],
    [_trail(0.0, 1024, 0, 2100, 0.8, 1.0), _trail(0.0, 1024, 1488, 2100, 6.4, 1.0),
     _trail(90.0, 0, 744, 1600, 0.9, 1.0), _trail(90.0, 2047, 744, 1600, 6.0, 1.0)],       # along the four edges
]


def test_rendering_matches_render_trails(bases, handles):
    hA, _ = handles
    rng = np.random.default_rng(7)
    slots = list(RENDER_SLOTS)
    while len(slots) < 40:
        slots.append(_random_grid(rng, int(rng.integers(1, 5))))
    bidx = np.arange(len(slots)) * 3 % B
    hA.submit_injected(bidx, slots)
    hA.wait()
    for j, ts in enumerate(slots):
        got = hA.stage(j, 0, "input")
        base = bases["frames"][bidx[j]]
        ref = render_trails(base.copy(), ts)
        cover = np.zeros((H, W), np.int32)
        peak = np.zeros((H, W), np.float32)
        for tr in ts:
            fp = footprint((H, W), tr)
            if fp is None:
                continue
            ya, yb, xa, xb, inside, _ = fp
            cover[ya:yb, xa:xb] += inside
            np.maximum(peak[ya:yb, xa:xb], np.where(inside, abs(np.float32(tr["peak"])), 0), out=peak[ya:yb, xa:xb])
        out = cover == 0
        assert np.array_equal(got[out].view(np.uint32), base[out].view(np.uint32)), "slot %d: pixels outside changed" % j
        ins = ~out
        mag = np.maximum(np.abs(ref[ins]), peak[ins])
        tol = 4 * cover[ins] * np.spacing(mag)
        err = np.abs(got[ins].astype(np.float64) - ref[ins].astype(np.float64))
        assert np.all(err <= tol), "slot %d: %d pixels beyond 4 ulps per trail (max %.3g)" % (j, int((err > tol).sum()), err.max())


def test_verdicts_and_production_path_match(bases, handles, cv2mod):
    """192 injections over the 64 bases: every device verdict is the oracle's on the downloaded input frame; the same
    frames through lfd_submit (graph path) on the other handle give byte-identical results, at B = 64 and n = 37."""
    hA, hB = handles
    kinds = bases["kinds"]
    assert any(k.startswith("dense") for k in kinds), "no dense field among the bases"
    rng = np.random.default_rng(192)
    grid = _random_grid(rng, 3 * B + 37)
    ndet = 0
    for k, n in enumerate((B, B, B, 37)):
        bidx = rng.permutation(B)[:n]
        slots = [[t] for t in grid[k * B:k * B + n]]
        for j in range(0, n, 9):
            slots[j].append(grid[(k * B + j + 100) % len(grid)])          # a few two-trail slots
        hA.submit_injected(bidx, slots)
        res = hA.wait()
        got = [device_verdict(r, (H, W)) for r in res]
        inj = [hA.stage(j, 0, "input") for j in range(n)]
        hB.submit(np.stack(inj), [bases["rects"][b] for b in bidx])
        res_b = hB.wait()
        assert [bytes(r) for r in res_b] == [bytes(r) for r in res], "batch %d (n = %d)" % (k, n)
        assert hA.counters()["ccl_lookback_stalls"] == 0 and hB.counters()["ccl_lookback_stalls"] == 0
        if k == 3:
            break                                                         # the ragged batch checks the production path only
        ref = verdicts(inj, [bases["cats"][b] for b in bidx], [bases["filters"][b] for b in bidx], PB, PD, PR)
        bad = ["slot %d (base %d, %s): got %s, oracle %s" % (j, bidx[j], kinds[bidx[j]], got[j], ref[j])
               for j in range(n) if got[j] != tuple(ref[j])]
        assert not bad, "\n".join(bad[:10])
        ndet += sum(1 for r in ref if r[0] is True)
    assert ndet >= 40, "grid too faint: only %d detections" % ndet
    # lfd_run_resident re-runs the injected frames of the last batch
    hA.run_resident(37)
    assert [bytes(r) for r in hA.wait()] == [bytes(r) for r in res_b]


def test_recovery_table(bases, cv2mod):
    sparse = [i for i, k in enumerate(bases["kinds"]) if k == "sparse"][:12]
    assert len(sparse) >= 8
    frames = bases["frames"][sparse]
    rects = [bases["rects"][i] for i in sparse]
    trail = {"p0": (100.0, 200.0), "p1": (1900.0, 1300.0), "sigma": 3.0, "peak": 3.0}
    rng = np.random.default_rng(5)
    injections = [(b, [trail]) for b in range(len(sparse))]
    injections += [(int(rng.integers(0, len(sparse))), _random_grid(rng, int(rng.integers(1, 3)))) for _ in range(70)]
    injections += [(0, [])]
    tab = recovery(frames, rects, injections, PB, PD, batch=32)
    assert len(tab) == len(injections)
    assert tab[-1]["recovered"] == -1 and tab[-1]["ntrails"] == 0
    for row, (b, ts) in zip(tab, injections):
        assert row["base"] == b and row["ntrails"] == len(ts)
        exp = -1
        if row["detected"] and not row["status"] & _lib.FRAME_OVERFLOW:
            hm = (PB, PD)[row["pass"]]["houghMethod"]
            for i, tr in enumerate(ts):
                rt, tt = trail_line(tr, (H, W))
                if any(abs(row["theta"] - tt - k * math.pi) <= np.deg2rad(2) and abs(row["rho"] - (-rt if k else rt)) <= hm
                       for k in (-1, 0, 1)):
                    exp = i
                    break
        assert row["recovered"] == exp
    # the oracle on the frames the device read (base + the synth `trail` geometry) decides where it must be recovered
    h = _lib.Handle(H, W, max_batch=len(sparse))
    try:
        h.set_params(PB, PD)
        h.set_base(frames, rects)
        h.submit_injected(np.arange(len(sparse)), [[trail]] * len(sparse))
        h.wait()
        inj = [h.stage(j, 0, "input") for j in range(len(sparse))]
    finally:
        h.close()
    ref = verdicts(inj, [bases["cats"][i] for i in sparse], [bases["filters"][i] for i in sparse], PB, PD, PR)
    hits = [j for j, r in enumerate(ref) if r[0] is True]
    assert hits, "the oracle detects the trail on none of the sparse bases"
    for j in hits:
        assert tab[j]["recovered"] == 0, (j, tab[j]["rho"], tab[j]["theta"], trail_line(trail, (H, W)))


def test_bad_input_launches_nothing():
    h = _lib.Handle(H, W, max_batch=4)
    rng = np.random.default_rng(3)
    frames = (rng.standard_normal((2, H, W), dtype=np.float32) * np.float32(0.025))
    frames[1] = synth.make_case("trail", 77)[0]
    try:
        h.set_params(PB, PD)

        def code(fn, *a, **k):
            with pytest.raises(_lib.LfdError) as e:
                fn(*a, **k)
            return e.value.code

        l0 = h.kernel_launches()
        assert code(h.submit_injected, [0]) == _lib.LFD_E_STATE                 # no base yet
        h.set_base(frames)
        ok = _trail(30.0, 1000, 700, 1000, 2.0, 3.0)
        assert code(h.submit_injected, []) == _lib.LFD_E_ARG                    # n = 0
        assert code(h.submit_injected, [0] * 5) == _lib.LFD_E_ARG               # n > B
        assert code(h.submit_injected, [0, 2]) == _lib.LFD_E_ARG                # base index out of range
        assert code(h.submit_injected, [-1]) == _lib.LFD_E_ARG
        assert code(h.submit_injected, [0], [[ok] * 17]) == _lib.LFD_E_ARG      # 17 trails in a slot
        for key, bad in (("p0", (math.nan, 1.0)), ("p1", (1.0, math.inf)), ("sigma", 0.0), ("sigma", -1.0),
                         ("sigma", math.nan), ("peak", math.inf)):
            assert code(h.submit_injected, [0, 1], [[ok], [dict(ok, **{key: bad})]]) == _lib.LFD_E_ARG, key
        assert code(h.submit_injected, [0], flags=_lib.INPUT_BIGENDIAN) == _lib.LFD_E_ARG
        assert h.kernel_launches() == l0, "a rejected call launched a kernel"
        # the handle still runs a valid batch, which equals the plain submit of the same frames
        h.submit_injected([1, 0], [[], []])
        got = [bytes(r) for r in h.wait()]
        h.submit(frames[::-1].copy())
        assert [bytes(r) for r in h.wait()] == got
        # after lfd_run_pass slot 0 holds a flipped frame: the input tap refuses
        h.run_pass(0, np.ascontiguousarray(frames[0][::-1]), writeback=False)
        assert code(h.stage, 0, 0, "input") == _lib.LFD_E_STATE
    finally:
        h.close()
