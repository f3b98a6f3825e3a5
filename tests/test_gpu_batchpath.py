"""Oracle parity of the PRODUCTION batch path - the one behind every number bench.py prints: lfd_submit with no tap
flags at B = 64 (CUDA graph, batch cut in two halves on four streams, two handles double-buffered), and the drop-in
driver DetectTrails(batch=32).process() on files.  Every frame's verdict (detected, pass, line end points) is compared
with oracle/ref_pipeline.py::process_frame (detecttrails.py:119-131 restated on cv2) on >= 256 frames of the config-3
mix (SURVEY.md 8(d)): trails at any angle incl. 0 / 90 degrees +- 1, widths 2-15 px, peaks 0.3-50, satellites, dense
fields up to 10 000 stars."""
import multiprocessing as mp
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from lfd_b200 import synth
from oracle import ref_pipeline as rp
from oracle.verdicts import device_verdict, verdicts

FORCED = ["trail_var", "trail_axis", "dense_heavy", "satellite", "faint_trail", "dense_trail", "trail", "dense"]


def _gen(job):
    kind, seed = job
    return synth.make_case(kind, seed)


def _pool(nmix, nforced):
    """(frames, cats, filters, kinds): nmix frames drawn like bench.py's pool + nforced frames of the hard kinds."""
    jobs, filters = [], []
    for i in range(nmix):
        flt = synth.FILTERS[i % 5]
        jobs.append(synth.case_for_frame(2888, 2, flt, 100 + i))
        filters.append(flt)
    for i in range(nforced):
        jobs.append((FORCED[i % len(FORCED)], 7000 + i))
        filters.append(synth.FILTERS[i % 5])
    with mp.get_context("fork").Pool(min(os.cpu_count() or 1, 32)) as pool:
        made = pool.map(_gen, jobs, chunksize=2)
    return [m[0] for m in made], [m[1] for m in made], filters, [j[0] for j in jobs]


def test_production_batches_match_oracle(cv2mod):
    from lfd_b200 import _lib
    from lfd_b200.removestars import star_rects
    B, NB = 64, 4
    frames, cats, filters, kinds = _pool(192, 64)
    assert len(frames) == B * NB
    pb, pd, pr = dict(rp.DEFAULT_BRIGHT), dict(rp.DEFAULT_DIM), dict(rp.DEFAULT_REMOVESTARS)
    ref = verdicts(frames, cats, filters, pb, pd, pr)
    rects = [star_rects(c, flt, f.shape, **{k: v for k, v in pr.items()}) for f, c, flt in zip(frames, cats, filters)]
    hs = [_lib.Handle(synth.FRAME_H, synth.FRAME_W, max_batch=B) for _ in range(2)]
    got = [None] * len(frames)
    try:
        for h in hs:
            h.set_params(pb, pd)

        def fill_and_submit(k):
            h = hs[k & 1]
            for j in range(B):
                h.host_frames[j] = frames[k * B + j]
            h.submit(B, rects[k * B:(k + 1) * B])           # no flags: graph + two halves + four streams

        def collect(k):
            h = hs[k & 1]
            res = h.wait()
            # the graph path records no per-stage events: all stage brackets behind k_prep read 0
            assert all(ms == 0.0 for _n, ms in h.timings()[2:]), "this batch did not take the CUDA-graph path"
            for j in range(B):
                got[k * B + j] = (device_verdict(res[j], frames[0].shape), bytes(res[j]))

        fill_and_submit(0)
        for k in range(1, NB):
            fill_and_submit(k)
            collect(k - 1)
        collect(NB - 1)
        bad = ["frame %d (%s, %s): got %s, oracle %s" % (i, kinds[i], filters[i], got[i][0], ref[i])
               for i in range(len(frames)) if got[i][0] != tuple(ref[i])]
        assert not bad, "%d of %d frames differ\n%s" % (len(bad), len(frames), "\n".join(bad[:20]))
        ndet = sum(1 for r in ref if r[0] is True)
        assert ndet >= 20, "pool too easy: only %d detections" % ndet
        assert {r[1] for r in ref if r[0] is True} == {0, 1}, "both passes must produce detections in this pool"
        # the resident re-run (bench.py's `value` leg) reproduces the last batch bit for bit
        h = hs[(NB - 1) & 1]
        h.run_resident(B)
        res2 = h.wait()
        for j in range(B):
            assert bytes(res2[j]) == got[(NB - 1) * B + j][1]
        # a ragged last batch (n = 37: halves of 19 and 18 frames) of frames the handle has not seen in these slots
        n = 37
        for j in range(n):
            h.host_frames[j] = frames[100 + j]
        h.submit(n, rects[100:100 + n])
        res3 = h.wait()
        for j in range(n):
            assert device_verdict(res3[j], frames[0].shape) == tuple(ref[100 + j]), (j, kinds[100 + j])
        # edge maps and box images the untapped (graph, batch parts) path left behind == the oracle's, pixel for pixel
        picked = [j for j in range(n) if ref[100 + j][0] is True][:3] + [j for j in range(n) if ref[100 + j][0] is False][:2]
        for j in picked:
            taps = {}
            rp.process_frame(frames[100 + j].copy(), cats[100 + j], filters[100 + j], taps=taps)
            for p, key in ((0, "bright"), (1, "dim")):
                if taps[key]:
                    assert np.array_equal(h.stage(j, p, "canny"), taps[key]["canny"]), (j, key, "canny")
                    assert np.array_equal(h.stage(j, p, "box"), taps[key]["box_img"]), (j, key, "box")
    finally:
        for h in hs:
            h.close()


def test_dropin_batches_match_oracle(tmp_path, cv2mod):
    """DetectTrails(batch=32).process() over 96 frames on disk (ring of three handles, loader threads, raw big-endian
    payload, native ingest) writes exactly the lines the oracle derives for the same files."""
    import lfd_b200
    from lfd_b200 import fitsio_lite
    fields = list(range(100, 196))
    kinds = {}
    for i, f in enumerate(fields):
        kinds[("r", f)] = FORCED[(i // 6) % len(FORCED)] if i % 6 == 0 else synth.case_for_frame(2888, 3, "r", f)[0]
    tree = synth.write_sdss_tree(str(tmp_path), 2888, 3, fields, filters=("r",), kinds=kinds, startfield=100, endfield=196)
    lfd_b200.setup(tree["bosspath"], tree["photoobjpath"], tree["photoreduxpath"], str(tmp_path))
    out = tmp_path / "out"
    out.mkdir()
    lfd_b200.DetectTrails(run=2888, camcol=3, filter="r", savepath=str(out), batch=32).process()
    got = (out / "results.txt").read_text()
    imgs = [tree["frames"][("r", f)][0] for f in fields]
    cats = [tree["frames"][("r", f)][1] for f in fields]
    ref = verdicts(imgs, cats, ["r"] * len(fields))
    exp = []
    for f, v in zip(fields, ref):
        if v[0] is True:
            path = os.path.join(tree["photoobjpath"], "frames", "301", "2888", "3", "frame-r-002888-3-%04d.fits" % f)
            exp.append(rp.result_line(2888, 3, "r", f, fitsio_lite.read_header(path), v[2]))
    assert got == "".join(exp)
    assert len(exp) >= 10
    assert (out / "errors.txt").read_text() == ""


def test_dropin_bz2_frames_and_overflow_retry(tmp_path, cv2mod, monkeypatch):
    """Compressed frames (detecttrails.py:81-111: `<frame>.fits.bz2` when the plain file is absent) go through the
    loader threads and the same staging slots as plain ones; a frame whose run / contour lists overflow the batch
    handles' capacities is re-run on a worst-case handle - either way results.txt is what the oracle derives and
    errors.txt stays empty."""
    import bz2
    import lfd_b200
    import lfd_b200.detecttrails as dtm
    from lfd_b200 import fitsio_lite
    fields = list(range(300, 312))
    names = ["trail_var", "dense_heavy", "sparse", "satellite", "dense", "trail", "sparse", "dense_trail", "faint_trail", "sparse",
             "trail_axis", "dense_heavy"]
    kinds = {("i", f): k for f, k in zip(fields, names)}
    tree = synth.write_sdss_tree(str(tmp_path), 2888, 4, fields, filters=("i",), kinds=kinds, startfield=300, endfield=312)
    fdir = os.path.join(tree["photoobjpath"], "frames", "301", "2888", "4")
    hdrs = {}
    for f in fields:
        path = os.path.join(fdir, "frame-i-002888-4-%04d.fits" % f)
        hdrs[f] = fitsio_lite.read_header(path)
        if f % 2 == 0:                                            # every other frame exists only compressed
            with open(path, "rb") as src, open(path + ".bz2", "wb") as dst:
                dst.write(bz2.compress(src.read(), 1))
            os.remove(path)
    lfd_b200.setup(tree["bosspath"], tree["photoobjpath"], tree["photoreduxpath"], str(tmp_path))
    ref = verdicts([tree["frames"][("i", f)][0] for f in fields], [tree["frames"][("i", f)][1] for f in fields], ["i"] * len(fields))
    exp = "".join(rp.result_line(2888, 4, "i", f, hdrs[f], v[2]) for f, v in zip(fields, ref) if v[0] is True)
    assert exp.count("\n") >= 4

    def run(tag):
        out = tmp_path / tag
        out.mkdir()
        lfd_b200.DetectTrails(run=2888, camcol=4, filter="i", savepath=str(out), batch=5).process()
        return (out / "results.txt").read_text(), (out / "errors.txt").read_text()

    assert run("plain") == (exp, "")
    # tiny work-list capacities: the dense fields overflow in the batch handles and are retried one by one
    monkeypatch.setenv("LFD_MAX_RUNS", "6000")
    monkeypatch.setenv("LFD_MAX_COMPONENTS", "600")
    calls = []
    real = dtm._big_handle
    monkeypatch.setattr(dtm, "_big_handle", lambda shape, device: (calls.append(shape), real(shape, device))[1])
    assert run("tiny") == (exp, "")
    assert len(calls) >= 2, "no frame overflowed: the retry path was not exercised"


def test_production_batch_config4_matches_oracle(cv2mod):
    """BASELINE.json config 4 through the production path (B = 64, no tap flags): high-sensitivity dim pass with a 15x15
    dilation kernel and rho = 1 px (numrho = 7075: two angles per vote CTA, per-pixel voting, single privatised copy);
    every verdict equals the oracle's with the same parameters."""
    from lfd_b200 import _lib
    from lfd_b200.removestars import star_rects
    B = 64
    frames, cats, filters, kinds = _pool(40, 24)
    pb = dict(rp.DEFAULT_BRIGHT)
    pd = dict(rp.DEFAULT_DIM, dilateKernel=np.ones((15, 15), np.uint8), houghMethod=1)
    pr = dict(rp.DEFAULT_REMOVESTARS)
    ref = verdicts(frames, cats, filters, pb, pd, pr)
    rects = [star_rects(c, flt, f.shape, **pr) for f, c, flt in zip(frames, cats, filters)]
    h = _lib.Handle(synth.FRAME_H, synth.FRAME_W, max_batch=B)
    try:
        h.set_params(pb, pd)
        for j in range(B):
            h.host_frames[j] = frames[j]
        h.submit(B, rects)
        res = h.wait()
        bad = ["frame %d (%s): got %s, oracle %s" % (i, kinds[i], device_verdict(res[i], frames[0].shape), ref[i])
               for i in range(B) if device_verdict(res[i], frames[0].shape) != tuple(ref[i])]
        assert not bad, "\n".join(bad[:10])
        assert sum(1 for r in ref if r[0] is True and r[1] == 1) >= 2, "no dim-pass detection in the pool"
    finally:
        h.close()
