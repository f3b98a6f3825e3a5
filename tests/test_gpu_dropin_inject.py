"""Injections in a drop-in run: lfd_capture_bases (k_capture_bases) makes a collected batch the injection bases, exactly,
from native and big-endian batches; it refuses every state in which the slots do not hold that batch; and
DetectTrails(injections=...) writes one line per injection that equals inject.recovery() on the same frames, leaves
results.txt / errors.txt / the progress file as they are without injections, and resumes without losing or repeating
a line."""
import math
import multiprocessing as mp
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from lfd_b200 import _lib, synth
from lfd_b200.inject import defocus_profile, read_injections, recovery
from oracle import ref_pipeline as rp
from test_gpu_inject_profiles import _check_slot

NB = 12
H, W = synth.FRAME_H, synth.FRAME_W
PB, PD, PR = dict(rp.DEFAULT_BRIGHT), dict(rp.DEFAULT_DIM), dict(rp.DEFAULT_REMOVESTARS)
TABLES = [defocus_profile(6.5, 2.6, 3.5),
          (0.0, 1.0, np.exp(-np.linspace(0.0, 3.0, 50)).astype(np.float32))]


def _gen(job):
    return synth.make_case(*job)


@pytest.fixture(scope="module")
def bases():
    from lfd_b200.removestars import star_rects
    jobs = [synth.case_for_frame(1336, 4, synth.FILTERS[i % 5], 60 + i) for i in range(NB)]
    filters = [synth.FILTERS[i % 5] for i in range(NB)]
    with mp.get_context("fork").Pool(min(os.cpu_count() or 1, NB)) as pool:
        made = pool.map(_gen, jobs, chunksize=1)
    frames = np.stack([m[0] for m in made])
    rects = [star_rects(m[1], flt, frames[0].shape, **PR) for m, flt in zip(made, filters)]
    return frames, rects


def _t(ang_deg, cx, cy, length, peak, sigma=2.0, profile=-1, lightcurve=-1):
    a = np.deg2rad(ang_deg)
    tr = {"p0": (float(np.float32(cx - length / 2 * math.cos(a))), float(np.float32(cy - length / 2 * math.sin(a)))),
          "p1": (float(np.float32(cx + length / 2 * math.cos(a))), float(np.float32(cy + length / 2 * math.sin(a)))),
          "sigma": float(np.float32(sigma)), "peak": float(np.float32(peak))}
    if profile >= 0:
        tr["profile"] = profile
        del tr["sigma"]
    if lightcurve >= 0:
        tr["lightcurve"] = lightcurve
    return tr


@pytest.mark.parametrize("big_endian", [False, True], ids=["native", "bigendian"])
def test_capture_is_exact(bases, big_endian):
    frames, rects = bases
    h = _lib.Handle(H, W, max_batch=NB)
    try:
        h.set_params(PB, PD)
        h.set_trail_tables(TABLES)
        if big_endian:
            h.submit(frames.byteswap(), rects, flags=_lib.INPUT_BIGENDIAN)
        else:
            h.submit(frames, rects)
        bare = [bytes(r) for r in h.wait()]
        h.capture_bases()
        # base b = slot b with its own rectangles: a permutation without trails gives the bare results permuted
        perm = np.arange(NB)[::-1].copy()
        h.submit_injected(perm)
        assert [bytes(r) for r in h.wait()] == [bare[b] for b in perm]
        kt = {k[0]: k for k in h.kernel_times()}
        assert kt["k_capture_bases"][2] > 0 and kt["k_capture_bases"][3] == 1
        h.submit_injected(np.arange(NB))
        assert [bytes(r) for r in h.wait()] == bare
        assert "k_capture_bases" not in {k[0] for k in h.kernel_times()}, "reported with a batch it did not precede"
        # with trails: the input tap is the native frame plus the reference rendering
        rng = np.random.default_rng(3)
        slots = []
        for j in range(NB):
            ts = [_t(rng.uniform(0, 180), rng.uniform(300, 1700), rng.uniform(300, 1200), rng.uniform(400, 2000),
                     rng.uniform(0.5, 20), sigma=rng.uniform(0.8, 6))]
            if j % 3 == 1:
                ts.append(_t(rng.uniform(0, 180), 1000, 700, 1500, 5.0, profile=0))
            if j % 3 == 2:
                ts.append(_t(rng.uniform(0, 180), 1000, 700, 1500, 5.0, profile=0, lightcurve=1))
            slots.append(ts)
        bidx = (np.arange(NB) * 5) % NB
        h.submit_injected(bidx, slots)
        h.wait()
        for j in range(NB):
            _check_slot(h.stage(j, 0, "input"), frames[bidx[j]], slots[j], TABLES, "slot %d" % j)
        # a ragged batch replaces the bases: only its n slots are bases now
        h.submit(frames[:5], rects[:5])
        h.wait()
        h.capture_bases()
        with pytest.raises(_lib.LfdError) as e:
            h.submit_injected([5])
        assert e.value.code == _lib.LFD_E_ARG
    finally:
        h.close()


def test_capture_refuses_states_without_the_batch(bases):
    frames, rects = bases
    h = _lib.Handle(H, W, max_batch=4)
    try:
        h.set_params(PB, PD)

        def refused():
            l0 = h.kernel_launches()
            with pytest.raises(_lib.LfdError) as e:
                h.capture_bases()
            assert e.value.code == _lib.LFD_E_STATE
            assert h.kernel_launches() == l0, "a refused capture launched a kernel"

        refused()                                                  # no batch yet
        h.submit(frames[:4], rects[:4])
        refused()                                                  # pending
        h.wait()
        h.capture_bases()
        h.submit_injected([0, 1], [[_t(30, 1000, 700, 1000, 3.0)], []])
        h.wait()
        refused()                                                  # the slots hold injected frames
        h.run_resident(2)
        h.wait()
        refused()                                                  # ... also after re-running them
        h.upload(frames[:2], rects[:2])                            # lfd_upload + lfd_run_resident: a batch again
        h.capture_bases()
        h.run_pass(0, np.ascontiguousarray(frames[0][::-1]), writeback=False)
        refused()                                                  # after lfd_run_pass
        h.submit(frames[:1], rects[:1])
        h.wait()
        j = max(range(NB), key=lambda i: len(rects[i]))
        assert len(rects[j]) > 0
        h.blot(frames[j].copy(), rects[j])
        refused()                                                  # after lfd_blot
    finally:
        h.close()


FIELDS = list(range(300, 312))
ODD_SHAPE_FIELD, ODD_H, ODD_W = 309, 1200, 1800
KINDS = ["trail_var", "dense_heavy", "sparse", "satellite", "dense", "trail", "sparse", "dense_trail", "faint_trail",
         "sparse", "trail_axis", "dense_heavy"]


def _injections(frame, shape):
    """Three injections per frame, deterministic in the frame: a bright Gaussian, a defocused trail without and one
    with a light curve next to a faint Gaussian."""
    h, w = shape
    rng = np.random.default_rng(synth.frame_seed(*frame) ^ 0x5eed)
    out = []
    for k in range(3):
        ang, cx, cy = rng.uniform(0, 180), rng.uniform(0.3 * w, 0.7 * w), rng.uniform(0.3 * h, 0.7 * h)
        if k == 0:
            out.append([_t(ang, cx, cy, rng.uniform(600, 2000), rng.uniform(0.5, 8.0), sigma=rng.uniform(0.8, 4.0))])
        else:
            out.append([_t(ang, cx, cy, rng.uniform(600, 2000), rng.uniform(0.5, 8.0), profile=0,
                           lightcurve=1 if k == 2 else -1)] +
                       ([_t(rng.uniform(0, 180), cx, cy, 800, 0.3, sigma=1.5)] if k == 2 else []))
    return out


@pytest.fixture(scope="module")
def tree(tmp_path_factory):
    """The drop-in tree of test_dropin_bz2_frames_and_overflow_retry, plus a missing frame file and a frame of another
    shape (it runs on a cached handle of its own)."""
    import bz2
    import lfd_b200
    from lfd_b200 import fitsio_lite
    root = tmp_path_factory.mktemp("tree")
    kinds = {("i", f): k for f, k in zip(FIELDS, KINDS)}
    t = synth.write_sdss_tree(str(root), 2888, 4, FIELDS, filters=("i",), kinds=kinds, startfield=300, endfield=312)
    fdir = os.path.join(t["photoobjpath"], "frames", "301", "2888", "4")
    for f in FIELDS:
        path = os.path.join(fdir, "frame-i-002888-4-%04d.fits" % f)
        if f == 305:
            os.remove(path)                                       # missing: an errors.txt entry, no injections
        elif f == ODD_SHAPE_FIELD:
            hdr = dict(synth.DEFAULT_HEADER, TAI=synth.DEFAULT_HEADER["TAI"] + f * 36.0)
            fitsio_lite.write_image(path, np.ascontiguousarray(t["frames"][("i", f)][0][:ODD_H, :ODD_W]), hdr)
        elif f % 2 == 0:
            with open(path, "rb") as src, open(path + ".bz2", "wb") as dst:
                dst.write(bz2.compress(src.read(), 1))
            os.remove(path)
    lfd_b200.setup(t["bosspath"], t["photoobjpath"], t["photoreduxpath"], str(root))
    return root


def _run(root, tag, **kw):
    import lfd_b200
    out = root / tag
    out.mkdir()
    lfd_b200.DetectTrails(run=2888, camcol=4, filter="i", savepath=str(out), batch=5, resume=True, **kw).process()
    return out


def _files(out):
    return [(out / n).read_text() for n in ("results.txt", "errors.txt", "progress.txt")]


def _recovery_rows(frames_ok):
    """inject.recovery() on the frames read by the reference's loaders, with the same injections and tables."""
    from lfd_b200.detecttrails import _load_frame
    from lfd_b200 import sdssfiles as files
    from lfd_b200.removestars import read_photoObj_arrays, star_rects
    groups, shapes = {}, []
    for i, fr in enumerate(frames_ok):
        img, _p = _load_frame(*fr)
        cat = read_photoObj_arrays(files.filename("photoObj", run=fr[0], camcol=fr[1], field=fr[3]))
        groups.setdefault(img.shape, []).append((i, img, star_rects(cat, fr[2], img.shape, **PR)))
        shapes.append(img.shape)
    rows = [None] * (3 * len(frames_ok))
    for shape, members in groups.items():              # one recovery() per frame shape
        jobs = [(b, ts) for b, (i, _img, _r) in enumerate(members) for ts in _injections(frames_ok[i], shape)]
        tab = recovery(np.stack([m[1] for m in members]), [m[2] for m in members], jobs, tables=TABLES)
        for b, (i, _img, _r) in enumerate(members):
            rows[3 * i:3 * i + 3] = tab[3 * b:3 * b + 3]
    return rows, shapes


def test_dropin_injections_equal_recovery(tree, monkeypatch):
    plain = _run(tree, "plain")
    inj = _run(tree, "inj", injections=_injections, injection_tables=TABLES)
    assert _files(inj) == _files(plain)
    assert "2888 4 i 305\n" in (plain / "errors.txt").read_text()
    tab = read_injections(str(inj / "injections.txt"))
    frames_ok = [(2888, 4, "i", f) for f in FIELDS if f != 305]
    assert len(tab) == 3 * len(frames_ok)
    ref, shapes = _recovery_rows(frames_ok)
    assert shapes.count((ODD_H, ODD_W)) == 1 and shapes.count((H, W)) == len(frames_ok) - 1
    detected = {tuple(ln.split()[:4]) for ln in (plain / "results.txt").read_text().splitlines()}
    for i, (row, rr) in enumerate(zip(tab, ref)):
        fr = frames_ok[i // 3]
        assert (int(row["run"]), int(row["camcol"]), str(row["filter"]), int(row["field"]), int(row["k"])) == fr + (i % 3,)
        ts = _injections(fr, shapes[i // 3])[i % 3]
        assert row["ntrails"] == rr["ntrails"] == len(ts)
        for f in ("x0", "y0", "x1", "y1", "sigma", "peak"):
            assert np.array_equal(row[f].view(np.uint32), rr[f].view(np.uint32)), (i, f)
        assert list(row["profile"][:len(ts)]) == [t.get("profile", -1) for t in ts]
        assert list(row["lightcurve"][:len(ts)]) == [t.get("lightcurve", -1) for t in ts]
        for f in ("detected", "pass", "status", "recovered"):
            assert row[f] == rr[f], (i, f, row[f], rr[f])
        assert row["rho"].view(np.uint32) == rr["rho"].view(np.uint32) and row["theta"].view(np.uint32) == rr["theta"].view(np.uint32), i
        assert row["base_detected"] == (tuple(str(v) for v in fr) in detected), i
    assert (tab["recovered"] >= 0).sum() >= 6 and (tab["recovered"] < 0).sum() >= 3, tab["recovered"]

    # tiny work lists: the dense fields' bare runs go to the overflow retry and keep their captured bases; injected
    # frames that overflow are reported in status; results.txt and the rest stay the run's without injections
    monkeypatch.setenv("LFD_MAX_RUNS", "6000")
    monkeypatch.setenv("LFD_MAX_COMPONENTS", "600")
    import lfd_b200.detecttrails as dtm
    calls = []
    real = dtm._big_handle
    monkeypatch.setattr(dtm, "_big_handle", lambda shape, device: (calls.append(shape), real(shape, device))[1])
    tiny = _run(tree, "tiny", injections=_injections, injection_tables=TABLES)
    assert len(calls) >= 2, "no frame overflowed: the retry path was not exercised"
    assert _files(tiny) == _files(plain)
    tt = read_injections(str(tiny / "injections.txt"))
    assert len(tt) == len(tab)
    over = (tt["status"] & _lib.FRAME_OVERFLOW) != 0
    assert over.any()
    assert np.all(tt["recovered"][over] == -1)
    assert np.array_equal(tt["base_detected"], tab["base_detected"])
    same = ~over
    for f in ("detected", "pass", "status", "recovered", "rho", "theta"):
        assert np.array_equal(tt[f][same], tab[f][same]), f


def test_resumed_run_writes_the_same_injection_table(tree):
    full = _run(tree, "full2", injections=_injections, injection_tables=TABLES)

    class Stop(Exception):
        pass

    def stopping(frame, shape):
        if frame[3] >= 310:                    # the sixth batch of two: at most the first four are written
            raise Stop()
        return _injections(frame, shape)

    import lfd_b200
    out = tree / "resumed"
    out.mkdir()
    kw = dict(run=2888, camcol=4, filter="i", savepath=str(out), batch=2, resume=True, injection_tables=TABLES)
    with pytest.raises(Stop):
        lfd_b200.DetectTrails(injections=stopping, **kw).process()
    part = (out / "injections.txt").read_text()
    assert 0 < part.count("\n") < (full / "injections.txt").read_text().count("\n")
    lfd_b200.DetectTrails(injections=_injections, **kw).process()
    assert (out / "injections.txt").read_text() == (full / "injections.txt").read_text()
    assert _files(out) == _files(full)
