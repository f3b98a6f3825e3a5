"""Run labelling on masks the synthetic pipeline inputs may not produce: a band over the shared-memory run capacity,
edges on the first and last column, widths that are not a multiple of 32, frames without candidates or without
selected edges, max_runs exactly at and one below the run count, and batches in which some passes overflow.

lfd_fit_min_area_rect runs Canny -> labelling straight on a uint8 image, so the edge map is what the image makes it;
the fg / bg label taps are then checked against the oracle's labelling of the edge map, and the run-id look-back of
the band kernel must never have given up waiting."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from lfd_b200 import synth
from oracle import cv_restate as cr
from oracle import ref_pipeline as rp


def _runs(mask):
    """runs of set pixels per row, summed over the rows"""
    m = np.pad(mask.astype(np.int8), ((0, 0), (1, 0)))
    return int((np.diff(m, axis=1) == 1).sum())


def _handle(H, W, max_runs=0):
    from lfd_b200 import _lib
    h = _lib.Handle(H, W, max_batch=1, max_runs=max_runs)
    h.set_params(dict(rp.DEFAULT_BRIGHT), dict(rp.DEFAULT_DIM))
    # lfd_get_stage reads frame slots of the last run: one pass makes slot 0 readable
    h.run_pass(0, np.zeros((H, W), np.float32), writeback=False)
    return h


def _labels(h, img):
    h.fit_min_area_rect(img, 1, 2, 1.0, 1.0)
    edges = h.stage(0, 0, "canny")
    return edges, h.stage(0, 0, "fg_labels"), h.stage(0, 0, "bg_labels")


def _check(h, img):
    edges, fg, bg = _labels(h, img)
    np.testing.assert_array_equal(fg, cr.label_fg8(edges))
    np.testing.assert_array_equal(bg, cr.label_bg4(edges))
    return edges


def _images(H, W):
    rng = np.random.default_rng(H * 7919 + W)
    out = {}
    # strong noise: thousands of runs per 32-row band (global union-find path)
    out["noise"] = (rng.random((H, W)) < 0.5).astype(np.uint8) * 255
    # outlined boxes, some cut by the first and the last column, one in the first and one in the last rows
    img = np.zeros((H, W), np.uint8)
    for (y0, x0, y1, x1) in ((5, 0, 40, 30), (60, W - 25, 120, W), (0, W // 3, 12, W // 3 + 50),
                             (H - 10, W // 2, H, W // 2 + 40), (H // 2, W // 4, H // 2 + 70, W // 4 + 90)):
        img[y0:y1, x0:x1] = 255
        img[y0 + 3:y1 - 3, max(x0 + 3, 0):x1 - 3] = 0
    img[:, 0] = np.where(np.arange(H) % 97 < 40, 255, 0)          # column 0 and column W-1 themselves
    img[:, W - 1] = np.where(np.arange(H) % 53 < 20, 255, 0)
    out["boxes"] = img
    # no candidates at all: one background run per row
    out["blank"] = np.zeros((H, W), np.uint8)
    # candidates without a single strong pixel: no selected edge, one background run per row
    out["weak"] = (rng.random((H, W)) < 0.01).astype(np.uint8) * 5
    return out


@pytest.mark.parametrize("H,W", [(synth.FRAME_H, synth.FRAME_W), (301, 1000), (97, 332), (64, 4096)])
def test_labels_match_oracle(H, W):
    h = _handle(H, W)
    try:
        for name, img in _images(H, W).items():
            if name == "noise" and H * W > 1 << 20:
                continue                                 # beyond the default contour capacities at this size
            edges = _check(h, img)
            if name in ("blank", "weak"):
                assert not edges.any(), name
            if name == "boxes":
                assert edges[:, 0].any() and edges[:, W - 1].any()
        if (H, W) == (64, 4096):
            # the noise image really has bands over the shared-memory capacity (CCL_BAND_CAP = 1536 runs per 32 rows)
            edges, _, _ = _labels(h, _images(H, W)["noise"])
            assert max(max(_runs(edges[y:y + 32] > 0), _runs(edges[y:y + 32] == 0)) for y in range(0, H, 32)) > 1536
    finally:
        h.close()


def test_max_runs_at_and_below_the_run_count():
    from lfd_b200 import _lib
    H, W = 256, 512
    img = _images(H, W)["boxes"]
    h = _handle(H, W)
    try:
        edges = _check(h, img)
    finally:
        h.close()
    nbg = _runs(edges == 0)                   # bg runs: every gap between selected fg runs
    assert _runs(edges > 0) < nbg
    h = _handle(H, W, max_runs=nbg)           # every run fits (the fg count is below the bg count)
    try:
        _check(h, img)
    finally:
        h.close()
    h = _handle(H, W, max_runs=nbg - 1)       # the hole pass has one run too many
    try:
        with pytest.raises(_lib.LfdError) as e:
            h.fit_min_area_rect(img, 1, 2, 1.0, 1.0)
        assert e.value.code == _lib.LFD_E_CAPACITY
        _check(h, _images(H, W)["blank"])     # the next call starts clean: H runs fit
    finally:
        h.close()


def test_batch_with_overflowing_passes():
    """A 24-frame batch (bands-looping CTAs, both passes and both halves concurrent) with a run capacity that some
    passes exceed: those frames report LFD_FRAME_OVERFLOW, every other frame is byte-identical to an unconstrained run."""
    from lfd_b200 import _lib
    from lfd_b200.removestars import star_rects
    kinds = ["trail", "sparse", "dense", "satellite", "faint_trail", "dense_trail", "empty", "sparse"]
    frames, rects = [], []
    for i in range(24):
        img, cat = synth.make_case(kinds[i % len(kinds)], 900 + i)
        frames.append(img)
        rects.append(star_rects(cat, "r", img.shape, **rp.DEFAULT_REMOVESTARS))
    frames = np.stack(frames)
    pb, pd = dict(rp.DEFAULT_BRIGHT), dict(rp.DEFAULT_DIM)
    res = {}
    for mr in (0, 6000):
        h = _lib.Handle(synth.FRAME_H, synth.FRAME_W, max_batch=24, max_runs=mr)
        try:
            h.set_params(pb, pd)
            for _ in range(2):                   # the second run replays the captured graph
                h.submit(frames, rects)
                out = h.wait()
                assert h.counters()["ccl_lookback_stalls"] == 0
            res[mr] = ([bytes(r) for r in out], [r.status for r in out])
        finally:
            h.close()
    over = [s & _lib.FRAME_OVERFLOW for s in res[6000][1]]
    assert 0 < sum(bool(o) for o in over) < 24
    assert not any(s & _lib.FRAME_OVERFLOW for s in res[0][1])
    for i in range(24):
        if not over[i]:
            assert res[6000][0][i] == res[0][0][i], i
