"""Structuring elements of any shape with sides up to 255 (lfd_set_kernels, k_morph_any's chord evaluation), bit-exact
against cv2 (oracle/ref_pipeline.py at the reference's call sites):

  stage parity   run_pass with LFD_KEEP_TAPS | LFD_FULL_LINES, both passes, on frames placed on k_morph_any's strip
                 and chunk seams (CHORD_SW, CHORD_R, read from the source) and an 8 x 8 frame; elements of >= 127 px
                 on small frames only, as cv2's tap-by-tap evaluation of them on a full frame takes seconds;
  production     the untapped batch path (CUDA graph, two batch parts) and the DetectTrails drop-in with a dim pass
                 of ellipse-5 erosion and ellipse-41 dilation, against oracle/verdicts.py;
  injection      recovery() with defocused-meteor trails and that element, against the oracle's verdict on the frame
                 tests/inject_shapes_ref.py::render_trails builds;
  limits         side 255 accepted, 256 refused, an empty element refused, and elements of different sizes one after
                 the other on one handle (graph rebuild, shared-memory opt-in)."""
import multiprocessing as mp
import os
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from lfd_b200 import synth
from oracle import ref_pipeline as rp
from oracle.verdicts import device_verdict, verdicts

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "lfd_b200", "csrc")
with open(os.path.join(CSRC, "k_morph.cuh")) as _f:
    _SRC = _f.read()
CHORD_SW = int(re.search(r"#define\s+CHORD_SW\s+(\d+)", _SRC).group(1))
CHORD_R = int(re.search(r"#define\s+CHORD_R\s+(\d+)", _SRC).group(1))
PROD = (synth.FRAME_H, synth.FRAME_W)
# frames on the strip and chunk seams (widths are multiples of 4, as lfd_create requires): one row and one word past a
# seam, exactly two chunks and strips, one row short of a chunk with W % 8 == 4 (the tile NMS kernel), and the smallest
SEAMS = [(CHORD_R + 1, CHORD_SW + 4), (2 * CHORD_R, 2 * CHORD_SW), (CHORD_R - 1, CHORD_SW + 12), (8, 8)]


def _ellipse(h, w=None):
    import cv2
    return cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (h if w is None else w, h))


def _cross(n):
    k = np.zeros((n, n), np.uint8)
    k[n // 2, :] = 1
    k[:, n // 2] = 1
    return k


def _ring(n, t):
    k = _ellipse(n)
    k[t:n - t, t:n - t] &= 1 - _ellipse(n - 2 * t)
    return k


def _ones(h, w):
    return np.ones((h, w), np.uint8)


# name: (bright dilate, dim erode, dim dilate, shapes)
CASES = {
    "ellipse41": (lambda: _ellipse(41), lambda: _ellipse(5), lambda: _ellipse(41), [PROD] + SEAMS),
    "ellipse63": (lambda: _ellipse(63), lambda: _ones(3, 3), lambda: _ellipse(63), [PROD] + SEAMS[:2]),
    "ellipse127": (lambda: _ellipse(127), lambda: _ellipse(5), lambda: _ellipse(127), SEAMS),
    "ellipse255": (lambda: _ellipse(255), lambda: _ellipse(9), lambda: _ellipse(255), SEAMS),
    "cross33": (lambda: _cross(33), lambda: _cross(3), lambda: _cross(33), [PROD] + SEAMS[:1]),
    "ring": (lambda: _ring(25, 4), lambda: _ones(3, 3), lambda: _ring(45, 6), [PROD] + SEAMS[:1]),
    "random40x37": (lambda: (np.random.default_rng(40).random((40, 37)) < 0.4).astype(np.uint8),
                    lambda: _ellipse(5), lambda: (np.random.default_rng(37).random((40, 37)) < 0.4).astype(np.uint8),
                    [PROD] + SEAMS[:1]),
    "ones64": (lambda: _ones(64, 64), lambda: _ones(3, 3), lambda: _ones(64, 64), [PROD] + SEAMS[:1]),
    "row255": (lambda: _ones(1, 255), lambda: _ones(1, 1), lambda: _ones(1, 255), SEAMS),
    "col255": (lambda: _ones(255, 1), lambda: _ones(3, 3), lambda: _ones(255, 1), SEAMS),
    "ellipse40x22": (lambda: _ellipse(40, 22), lambda: _ellipse(4, 6), lambda: _ellipse(40, 22), [PROD] + SEAMS[:2]),
    "erode33_dilate65": (lambda: _ellipse(9), lambda: _ellipse(33), lambda: _ellipse(65), [PROD] + SEAMS[:2]),
}
STAGE_CASES = [(name, shape) for name, c in CASES.items() for shape in c[3]]


def _params(name, shape):
    bd, ee, dd, _ = CASES[name]
    lw = 5 if min(shape) >= 64 else 1              # lets a streak pass in the tiny frames too
    pb = dict(rp.DEFAULT_BRIGHT, dilateKernel=bd(), lwTresh=lw)
    pd = dict(rp.DEFAULT_DIM, erodeKernel=ee(), dilateKernel=dd(), lwTresh=lw)
    return pb, pd


def _frame(shape, seed):
    H, W = shape
    if shape == PROD:
        img, _ = synth.make_case("trail", seed)
        return img
    return synth.make_frame(seed, n_stars=max(2, H * W // 4000), h=H, w=W, trails=[
        {"p0": (0.1 * W, 0.2 * H), "p1": (0.9 * W, 0.85 * H), "sigma": 2.5, "peak": 2.0}])[0]


def _check(h, pass_, work, params, tag):
    from lfd_b200 import _lib
    from lfd_b200.processfield import result_from_device
    ref_img = work.copy()
    taps = {}
    ref_res = (rp.bright_pass if pass_ == 0 else rp.dim_pass)(ref_img, taps=taps, **params)
    r = h.run_pass(pass_, work, flags=_lib.KEEP_TAPS | _lib.FULL_LINES, writeback=True)
    errs = []
    for stage, key in (("gray", "gray"), ("equ", "equ"), ("morph", "morph"), ("canny", "canny"), ("box", "box_img")):
        got = h.stage(0, pass_, stage)
        if not np.array_equal(got, taps[key]):
            errs.append("%s: %d px differ" % (stage, int((got != taps[key]).sum())))
    if pass_ == 1 and params.get("erodeKernel") is not None:
        if not np.array_equal(h.stage(0, pass_, "eroded"), taps["eroded"]):
            errs.append("eroded")
    rects = [a for a in h.stage(0, pass_, "rects") if a["kind"] != 2]
    if len(rects) != len(taps["rects"]):
        errs.append("contours: %d vs %d from cv2" % (len(rects), len(taps["rects"])))
    gp = sorted(((float(a["cx"]), float(a["cy"])), (float(a["w"]), float(a["h"])), float(a["angle"])) for a in rects if a["passed"])
    if gp != sorted(x for x, _ in taps["passing"]):
        errs.append("passing rects differ: %d vs %d" % (len(gp), len(taps["passing"])))
    if taps["passing"]:
        for which, key in (("equ", "lines_equ"), ("box", "lines_box")):
            ref_lines, got_lines = taps[key], h.stage(0, pass_, "lines_" + which)
            if ref_lines is None:
                if len(got_lines):
                    errs.append("lines_%s: expected none" % which)
            elif got_lines.shape != ref_lines.shape or not np.array_equal(got_lines.view(np.uint32), ref_lines.view(np.uint32)):
                errs.append("lines_%s: %s vs %s" % (which, got_lines.shape, ref_lines.shape))
    assert not errs, "%s pass %d: %s" % (tag, pass_, "; ".join(errs))
    assert result_from_device(r, pass_, work.shape) == ref_res
    return len(taps["passing"])


@pytest.mark.parametrize("name,shape", STAGE_CASES, ids=["%s-%dx%d" % (n, s[0], s[1]) for n, s in STAGE_CASES])
def test_stage_parity(cv2mod, name, shape):
    from lfd_b200 import _lib
    pb, pd = _params(name, shape)
    h = _lib.Handle(shape[0], shape[1], max_batch=1)
    try:
        h.set_params(pb, pd)
        work = np.ascontiguousarray(_frame(shape, 31)[::-1])
        _check(h, 0, work.copy(), pb, name)
        w1 = work.copy()
        w1[w1 < 0] = 0
        _check(h, 1, w1, pd, name)
    finally:
        h.close()


def _gen(job):
    return synth.make_case(*job)


@pytest.fixture(scope="module")
def pool():
    """37 config-3 frames (bench.py's mix) with catalogs, filters and star rectangles."""
    from lfd_b200.removestars import star_rects
    jobs = [synth.case_for_frame(2888, 5, synth.FILTERS[i % 5], 300 + i) for i in range(37)]
    filters = [synth.FILTERS[i % 5] for i in range(37)]
    with mp.get_context("fork").Pool(min(os.cpu_count() or 1, 32)) as p:
        made = p.map(_gen, jobs, chunksize=1)
    frames = [m[0] for m in made]
    cats = [m[1] for m in made]
    rects = [star_rects(c, flt, frames[0].shape, **rp.DEFAULT_REMOVESTARS) for c, flt in zip(cats, filters)]
    return {"frames": frames, "cats": cats, "filters": filters, "rects": rects, "kinds": [j[0] for j in jobs]}


def _dim41():
    return dict(rp.DEFAULT_DIM, erodeKernel=_ellipse(5), dilateKernel=_ellipse(41))


def test_production_batch(pool, cv2mod):
    from lfd_b200 import _lib
    pb, pd = dict(rp.DEFAULT_BRIGHT), _dim41()
    frames, n = pool["frames"], len(pool["frames"])
    ref = verdicts(frames, pool["cats"], pool["filters"], pb, pd, dict(rp.DEFAULT_REMOVESTARS))
    h = _lib.Handle(synth.FRAME_H, synth.FRAME_W, max_batch=64)
    try:
        h.set_params(pb, pd)
        for j in range(n):
            h.host_frames[j] = frames[j]
        h.submit(n, pool["rects"])                              # no flags: CUDA graph, two batch parts
        res = h.wait()
        assert all(ms == 0.0 for _n, ms in h.timings()[2:]), "this batch did not take the CUDA-graph path"
        got = [device_verdict(res[j], frames[0].shape) for j in range(n)]
        bad = ["frame %d (%s): got %s, oracle %s" % (j, pool["kinds"][j], got[j], ref[j]) for j in range(n) if got[j] != tuple(ref[j])]
        assert not bad, "\n".join(bad[:10])
        assert sum(1 for r in ref if r[0] is True) >= 2, "pool too easy"
    finally:
        h.close()


def test_detecttrails_dropin(tmp_path, cv2mod):
    import lfd_b200
    from lfd_b200 import fitsio_lite
    fields = [100, 101, 102, 103, 104]
    kinds = {("r", 100): "faint_trail", ("r", 101): "sparse", ("r", 102): "trail", ("r", 103): "dense_trail",
             ("r", 104): "faint_trail"}
    tree = synth.write_sdss_tree(str(tmp_path), 2888, 1, fields, filters=("r",), kinds=kinds, startfield=100, endfield=105)
    lfd_b200.setup(tree["bosspath"], tree["photoobjpath"], tree["photoreduxpath"], str(tmp_path))
    out = tmp_path / "out"
    out.mkdir()
    dt = lfd_b200.DetectTrails(run=2888, camcol=1, filter="r", savepath=str(out), batch=3)
    dt.params_dim["erodeKernel"] = _ellipse(5)
    dt.params_dim["dilateKernel"] = _ellipse(41)
    dt.process()
    pd = _dim41()
    exp = []
    for field in fields:
        path = os.path.join(tree["photoobjpath"], "frames", "301", "2888", "1", "frame-r-002888-1-%04d.fits" % field)
        det, _p, res = rp.process_frame(fitsio_lite.read(path), tree["frames"][("r", field)][1], "r", params_dim=pd)
        if det:
            exp.append(rp.result_line(2888, 1, "r", field, fitsio_lite.read_header(path), res))
    assert (out / "errors.txt").read_text() == ""
    assert (out / "results.txt").read_text() == "".join(exp)
    assert exp


def test_recovery_defocused(pool, cv2mod):
    from lfd_b200.inject import defocus_profile, recovery
    from inject_shapes_ref import render_trails
    sparse = [i for i, k in enumerate(pool["kinds"]) if k == "sparse"][:4]
    assert len(sparse) >= 2
    frames = np.stack([pool["frames"][i] for i in sparse])
    rects = [pool["rects"][i] for i in sparse]
    tables = [defocus_profile(8.0, 3.2, 3.5), defocus_profile(12.0, 4.8, 3.5)]
    injections = []
    for b in range(len(sparse)):
        for pk in (0.1, 0.5):
            injections.append((b, [{"p0": (100.0, 200.0 + 50 * b), "p1": (1900.0, 1300.0), "peak": pk, "profile": 1}]))
        injections.append((b, [{"p0": (300.0, 1400.0), "p1": (1700.0, 90.0 + 40 * b), "peak": 0.8, "profile": 0}]))
    pb, pd = dict(rp.DEFAULT_BRIGHT), _dim41()
    tab = recovery(frames, rects, injections, pb, pd, batch=8, tables=tables)
    inj = [render_trails(frames[b].copy(), ts, tables) for b, ts in injections]
    ref = verdicts(inj, [pool["cats"][sparse[b]] for b, _ in injections], [pool["filters"][sparse[b]] for b, _ in injections],
                   pb, pd, dict(rp.DEFAULT_REMOVESTARS))
    for j, r in enumerate(ref):
        assert bool(tab[j]["detected"]) == (r[0] is True), (j, r)
        if r[0] is True:
            assert tab[j]["pass"] == r[1], (j, r)
    assert any(r[0] is True for r in ref), "no injection detected"


def test_limits_and_switching(cv2mod):
    from lfd_b200 import _lib
    shape = SEAMS[0]
    frames = np.stack([_frame(shape, s) for s in (3, 4, 5)])
    h = _lib.Handle(shape[0], shape[1], max_batch=4)
    try:
        pb = dict(rp.DEFAULT_BRIGHT, lwTresh=2)
        for dk in (_ellipse(255), _ellipse(255, 1), _ones(255, 255)):
            h.set_params(pb, dict(rp.DEFAULT_DIM, dilateKernel=dk))
        for bad in (_ellipse(256), _ones(1, 256), _ones(256, 3)):
            with pytest.raises(_lib.UnsupportedParameter, match="1..255"):
                h.set_params(pb, dict(rp.DEFAULT_DIM, dilateKernel=bad))
            with pytest.raises(_lib.UnsupportedParameter, match="1..255"):
                h.set_params(pb, dict(rp.DEFAULT_DIM, erodeKernel=bad, dilateKernel=_ellipse(9)))
        with pytest.raises(_lib.LfdError) as ei:
            h.set_params(pb, dict(rp.DEFAULT_DIM, dilateKernel=np.zeros((7, 7), np.uint8)))
        assert ei.value.code == _lib.LFD_E_ARG
        # small -> 255 -> small on one handle, each through the graph path and against the oracle
        for dk, ek in ((_ellipse(9), _ellipse(3)), (_ellipse(255), _ellipse(41)), (_cross(7), _ellipse(3)),
                       (_ellipse(127), _ones(1, 1))):
            pd = dict(rp.DEFAULT_DIM, erodeKernel=ek, dilateKernel=dk, lwTresh=2)
            pbk = dict(pb, dilateKernel=dk)
            h.set_params(pbk, pd)
            for rep in range(2):
                h.submit(frames)
                res = h.wait()
                assert all(ms == 0.0 for _n, ms in h.timings()[2:])
                for j in range(len(frames)):
                    exp = rp.process_frame(frames[j].copy(), None, "r", pbk, pd)
                    assert device_verdict(res[j], shape) == tuple(exp), (dk.shape, j, rep)
    finally:
        h.close()
