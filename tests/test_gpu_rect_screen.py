"""k_rects_screen on the device: its verdicts against the NumPy restatement of tests/test_rect_screen_cpu.py, its rejected
contours against their fitted rectangles (LFD_KEEP_TAPS fits every contour), and the production path (no taps: CUDA
graph, two batch parts, only the survivors fitted) against the oracle and against the tapped run of the same frames."""
import multiprocessing as mp
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from lfd_b200 import synth
from oracle import cv_restate as cr
from oracle import ref_pipeline as rp
from oracle.verdicts import device_verdict, verdicts
from test_rect_screen_cpu import passes, screen_rejects

CONFIGS = ("config3", "config4")


def _gen(job):
    return synth.make_case(*job)


@pytest.fixture(scope="module")
def pool():
    """256 + 37 frames drawn like bench.py's pool (run 2888, camcol 1, fields 11 ..), with their blot rectangles."""
    from lfd_b200.removestars import star_rects
    n = 256 + 37
    filters = [synth.FILTERS[i % 5] for i in range(n)]
    jobs = [synth.case_for_frame(2888, 1, filters[i], 11 + i) for i in range(n)]
    with mp.get_context("fork").Pool(min(os.cpu_count() or 1, 32)) as p:
        made = p.map(_gen, jobs, chunksize=2)
    pr = {k: v for k, v in rp.DEFAULT_REMOVESTARS.items() if k != "debug"}
    frames = [m[0] for m in made]
    cats = [m[1] for m in made]
    rects = [star_rects(c, flt, f.shape, **pr) for f, c, flt in zip(frames, cats, filters)]
    return frames, cats, filters, rects


def _params(config):
    """bench.py's parameters: config 3 = the defaults, config 4 = 15 x 15 dilation and houghMethod 1 in the dim pass."""
    pb, pd = dict(rp.DEFAULT_BRIGHT), dict(rp.DEFAULT_DIM)
    if config == "config4":
        pd = dict(pd, dilateKernel=np.ones((15, 15), np.uint8), houghMethod=1.0)
    return pb, pd


def _run(h, frames, rects, flags):
    for j, f in enumerate(frames):
        h.host_frames[j] = f
    h.submit(len(frames), rects, flags=flags)
    return h.wait()


def _by_key(h, n):
    """{(frame, pass): {key: (record, screened)}} of the RECTS and RECT_SCREEN taps (edge-pixel and hole-pixel keys are
    disjoint, so the key alone names a contour)."""
    out = {}
    for f in range(n):
        for p in (0, 1):
            rects, scr = h.stage(f, p, "rects"), h.stage(f, p, "rect_screen")
            assert len(rects) == len(scr)
            out[(f, p)] = {int(o["key"]): (o, int(s)) for o, s in zip(rects, scr)}
            assert len(out[(f, p)]) == len(rects)
    return out


@pytest.mark.parametrize("config", CONFIGS)
def test_screen_verdicts_under_taps(cv2mod, pool, config):
    """KEEP_TAPS, 24 frames: the device's verdict for every contour of both passes equals the restatement on the
    structural point set of the pass's CANNY tap; every rejected contour's fitted rectangle fails the length/width
    filter; the counter rects_screened is the number of rejections."""
    from lfd_b200 import _lib
    frames, _cats, _flt, rects = pool
    pb, pd = _params(config)
    n = 24
    h = _lib.Handle(synth.FRAME_H, synth.FRAME_W, max_batch=n)
    try:
        h.set_params(pb, pd)
        _run(h, frames[:n], rects[:n], _lib.KEEP_TAPS)
        counted = h.counters()["rects_screened"]
        total = rejected = 0
        for f in range(n):
            for p, pp in ((0, pb), (1, pd)):
                recs, scr = h.stage(f, p, "rects"), h.stage(f, p, "rect_screen")
                sets = {key: pts for _k, key, pts in cr.contour_point_sets(h.stage(f, p, "canny"))}
                assert len(sets) == len(recs), (f, p)
                for o, s in zip(recs, scr):
                    want = screen_rejects(sets[int(o["key"])], pp["lwTresh"])
                    assert bool(s) == want, (f, p, int(o["kind"]), int(o["key"]))
                    if s:
                        assert int(o["passed"]) == 0 and int(o["kind"]) in (0, 1)
                        assert not passes(((o["cx"], o["cy"]), (float(o["w"]), float(o["h"])), o["angle"]),
                                          pp["minAreaRectMinLen"], pp["lwTresh"])
                total += len(recs)
                rejected += int(scr.sum())
        print("%s: %d contours, %d screened" % (config, total, rejected))
        assert counted == rejected and rejected > 0.9 * total
    finally:
        h.close()


@pytest.mark.parametrize("config", CONFIGS)
def test_production_path_matches_oracle_and_taps(cv2mod, pool, config):
    """256 + 37 frames in batches of 64 (the last one 37): the production path (no flags: CUDA graph, two batch parts)
    gives every frame the oracle's verdict and line.  Against a KEEP_TAPS run of the same batch: the same screened and
    contour counters, the same verdict per contour, the rejected contours recorded as kind 3 without a fit, every
    survivor's record identical to its fit in the tapped run, and the same results."""
    from lfd_b200 import _lib
    frames, cats, filters, rects = pool
    pb, pd = _params(config)
    pr = dict(rp.DEFAULT_REMOVESTARS)
    ref = verdicts(frames, cats, filters, pb, pd, pr)
    h = _lib.Handle(synth.FRAME_H, synth.FRAME_W, max_batch=64)
    bad = []
    try:
        h.set_params(pb, pd)
        for b0 in range(0, len(frames), 64):
            fr, rc = frames[b0:b0 + 64], rects[b0:b0 + 64]
            n = len(fr)
            res = _run(h, fr, rc, 0)
            assert all(ms == 0.0 for _n, ms in h.timings()[2:]), "this batch did not take the CUDA-graph path"
            for j in range(n):
                v = device_verdict(res[j], frames[0].shape)
                if v != tuple(ref[b0 + j]):
                    bad.append("frame %d: got %s, oracle %s" % (b0 + j, v, ref[b0 + j]))
            prod_res = [bytes(r) for r in res[:n]]
            prod_cnt = h.counters()
            prod = _by_key(h, n)
            res_t = _run(h, fr, rc, _lib.KEEP_TAPS)
            tap_cnt = h.counters()
            tap = _by_key(h, n)
            assert [bytes(r) for r in res_t[:n]] == prod_res, b0
            for k in ("rects_screened", "contours", "passing_rects", "frames_hough"):
                assert prod_cnt[k] == tap_cnt[k], (b0, k, prod_cnt[k], tap_cnt[k])
            assert prod_cnt["rects_screened"] > 0.9 * prod_cnt["contours"]
            for fp, recs in prod.items():
                assert recs.keys() == tap[fp].keys(), fp
                for key, (o, s) in recs.items():
                    ot, st = tap[fp][key]
                    assert s == st, (b0, fp, key)
                    if s:
                        assert int(o["kind"]) == 3 and int(o["passed"]) == 0, (b0, fp, key)
                    else:
                        assert o.tobytes() == ot.tobytes(), (b0, fp, key)
        assert not bad, "%d of %d frames differ\n%s" % (len(bad), len(frames), "\n".join(bad[:20]))
        assert sum(1 for r in ref if r[0] is True) >= 10
    finally:
        h.close()
