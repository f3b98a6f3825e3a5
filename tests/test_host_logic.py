"""CPU tests of the host side: catalog filter, FITS stand-in, path templating, DetectTrails selection logic,
result decoding, and the C-ABI library's symbols (no compute calls without a GPU)."""
import ctypes
import os

import numpy as np
import pytest

import lfd_b200
from lfd_b200 import _lib, fitsio_lite, sdssfiles, synth
from lfd_b200.removestars import star_rects
from oracle import ref_pipeline as rp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def test_abi_library_exports_header_symbols():
    import __graft_entry__ as ge
    ge.build()
    L = ctypes.CDLL(_lib.LIB_PATH)
    syms = ge.exported_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(L, s), s
    assert L.lfd_abi_version() == 1
    # struct layout agreed between header and ctypes
    assert ctypes.sizeof(_lib.PassParams) == 8 * 8 + 8 * 4
    assert ctypes.sizeof(_lib.Result) == 4 * 3 + 4 * 8 + 8 + 2 * 2 * 16 * 2 * 4
    assert _lib.RECT_DTYPE.itemsize == 5 * 4 + 3 * 4 + 8 * 4


def test_no_gpu_fails_loudly():
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("GPU present")
    except ImportError:
        pass
    with pytest.raises(_lib.LfdError):
        _lib.Handle(64, 64)


@pytest.mark.parametrize("flt", list("ugriz"))
def test_star_rects_match_oracle(flt):
    for seed in (1, 2, 3):
        img, cat = synth.make_case("sparse", seed)
        ref = rp.star_rects(cat, flt, **rp.DEFAULT_REMOVESTARS)
        a = np.ones(img.shape, np.float32)
        rp.blot(a, ref)
        b = np.ones(img.shape, np.float32)
        for r0, r1, c0, c1 in star_rects(cat, flt, img.shape, **rp.DEFAULT_REMOVESTARS):
            b[r0:r1, c0:c1] = 0
        assert np.array_equal(a, b)
        assert (a == 0).any()


def test_star_rects_nan_raises_like_math_ceil():
    _img, cat = synth.make_case("sparse", 4)
    cat["ROWC"][3, 2] = np.nan
    with pytest.raises(ValueError):
        star_rects(cat, "r", (1489, 2048), **rp.DEFAULT_REMOVESTARS)


def test_fitsio_lite_roundtrip(tmp_path):
    img = np.random.default_rng(0).normal(size=(37, 52)).astype(np.float32)
    p = str(tmp_path / "a.fits")
    fitsio_lite.write_image(p, img, dict(synth.DEFAULT_HEADER))
    assert np.array_equal(fitsio_lite.read(p), img)
    h = fitsio_lite.read_header(p)
    assert h["TAI"] == synth.DEFAULT_HEADER["TAI"] and h["NAXIS1"] == 52
    raw, _ = fitsio_lite.read_raw_image(p)
    assert np.array_equal(raw.view(">f4").astype(np.float32), img)
    _img, cat = synth.make_case("sparse", 5)
    q = str(tmp_path / "b.fits")
    fitsio_lite.write_bintable(q, cat)
    data, hdr = fitsio_lite.read(q, header="True")
    assert hdr["XTENSION"] == "BINTABLE"
    for k in cat:
        assert np.array_equal(data[k], cat[k]), k


def test_paths_and_runlist(tmp_path):
    tree = synth.write_sdss_tree(str(tmp_path), 2888, 3, [10], filters=("i",), kinds="empty")
    lfd_b200.setup(tree["bosspath"], tree["photoobjpath"], tree["photoreduxpath"], str(tmp_path))
    f = sdssfiles.filename("frame", run=2888, camcol=3, field=10, filter="i")
    assert f.endswith("frames/301/2888/3/frame-i-002888-3-0010.fits") and os.path.exists(f)
    o = sdssfiles.filename("photoObj", run=2888, camcol=3, field=10)
    assert o.endswith("301/2888/3/photoObj-002888-3-0010.fits") and os.path.exists(o)
    with pytest.raises(ValueError):
        sdssfiles.filename("frame", run=1, camcol=3, field=10, filter="i")


def test_frame_order_matches_reference(tmp_path):
    g = np.load(os.path.join(GOLD, "golden_run.npz"))
    tree = synth.write_sdss_tree(str(tmp_path), 2888, 1, [100], filters=("r",), kinds="empty", startfield=100, endfield=103)
    lfd_b200.setup(tree["bosspath"], tree["photoobjpath"], tree["photoreduxpath"], str(tmp_path))
    for name, kw in (("run", dict(run=2888)), ("run-camcol", dict(run=2888, camcol=2)),
                     ("run-filter", dict(run=2888, filter="i")), ("run-camcol-filter", dict(run=2888, camcol=3, filter="z")),
                     ("camcol-filter", dict(camcol=4, filter="u")), ("camcol-frame", dict(run=2888, camcol=5, field=101)),
                     ("field", dict(run=2888, camcol=6, filter="g", field=102))):
        d = lfd_b200.DetectTrails(**kw)
        assert d._pick == name
        got = np.array([(r, c, "ugriz".index(f), fl) for r, c, f, fl in d.frame_list()], np.int64).reshape(-1, 4)
        assert np.array_equal(got, g["order_" + name]), name


def test_constructor_quirks():
    pb, pd, pr = lfd_b200.default_params()
    d = lfd_b200.DetectTrails(run=1, params_dim={"debug": False, "x": 1})
    assert d.params_bright == {"debug": False, "x": 1}          # reference bug kept (detecttrails.py:253-254)
    assert set(d.params_dim) == set(pd) and set(d.params_removestars) == set(pr)
    with pytest.raises(ValueError):
        lfd_b200.DetectTrails(camcol=9)
    with pytest.raises(ValueError):
        lfd_b200.DetectTrails(run=1, field=3)
    assert lfd_b200.DetectTrails(run=1, camcol=1, savepath="/x").results == "/x/results.txt"


def test_result_decoding():
    from lfd_b200.processfield import result_from_device
    r = _lib.Result()
    r.rect_detection[0] = 0
    assert result_from_device(r, 0, (1489, 2048)) == (False, None)
    r.rect_detection[0] = 1
    r.rejected[0] = 1
    assert result_from_device(r, 0, (1489, 2048)) == (False, None)
    r.rejected[0] = 0
    r.top_equ[0][0][0] = 1180.0
    r.top_equ[0][0][1] = np.float32(1.0122910)
    got = result_from_device(r, 0, (1489, 2048))
    assert got == (True, rp.dictify_hough((1489, 2048), (np.float32(1180.0), np.float32(1.0122910))))
    r.status = _lib.FRAME_NO_LINES_BOX
    with pytest.raises(TypeError):
        result_from_device(r, 0, (1489, 2048))


def test_kernel_shapes_are_passed_through():
    pb, pd, _ = lfd_b200.default_params()
    cross = dict(pd, erodeKernel=np.array([[0, 1, 0], [1, 1, 1], [0, 1, 0]], np.uint8))
    p = _lib.pass_params(cross, True)              # a cross is legal: it goes to lfd_set_kernels at set_params time
    assert (p.erode_h, p.erode_w, p.dilate_h, p.dilate_w) == (3, 3, 9, 9)
    assert not _lib._all_ones(cross["erodeKernel"]) and _lib._all_ones(pd["dilateKernel"])
    with pytest.raises(ValueError):
        _lib.pass_params(dict(pd, dilateKernel=np.ones(5, np.uint8)), True)


def test_check_theta_matches_oracle():
    rng = np.random.default_rng(1)
    for _ in range(200):
        n1, n2 = rng.integers(1, 6, 2)
        h1 = np.stack([rng.integers(-50, 50, n1) * 20.0, rng.integers(0, 180, n1) * np.float32(np.pi / 180)], 1).astype(np.float32).reshape(n1, 1, 2)
        h2 = np.stack([rng.integers(-50, 50, n2) * 20.0, rng.integers(0, 180, n2) * np.float32(np.pi / 180)], 1).astype(np.float32).reshape(n2, 1, 2)
        if rng.random() < 0.5:
            h2[:, 0, :] = h1[:1, 0, :] + rng.normal(0, 0.05, (n2, 2)).astype(np.float32)
        assert lfd_b200.check_theta(h1, h2, 3, 25, 0.15, 0.15, False) == rp.check_theta(h1, h2, 3, 25, 0.15, 0.15)


def test_star_rects_batch_equals_per_frame():
    """The batched catalog filter (one set of NumPy calls per GPU batch) returns exactly the per-frame rectangles,
    for mixed filters, an empty catalog and a catalog with a NaN (which only fails its own frame)."""
    from lfd_b200.removestars import star_rects_batch
    cats, flts = [], []
    for i, flt in enumerate("ugrizrg"):
        _img, cat = synth.make_case("dense" if i % 3 == 0 else "sparse", 70 + i)
        cats.append(cat); flts.append(flt)
    empty = {k: np.asarray(v)[:0] for k, v in cats[0].items()}
    bad = {k: np.array(v, copy=True) for k, v in cats[1].items()}
    bad["PSFMAG"] = bad["PSFMAG"].astype(np.float32); bad["PSFMAG"][3, 2] = np.nan
    exc = OSError("unreadable photoObj")
    for batch, fl in ((cats, flts), (cats[:2] + [empty] + cats[2:], flts[:2] + ["r"] + flts[2:]),
                      (cats[:3] + [bad, exc] + cats[3:], flts[:3] + ["i", "z"] + flts[3:])):
        got = star_rects_batch(batch, fl, (1489, 2048), **rp.DEFAULT_REMOVESTARS)
        assert len(got) == len(batch)
        for c, f, g in zip(batch, fl, got):
            if isinstance(c, BaseException):
                assert g is c
                continue
            try:
                ref = star_rects(c, f, (1489, 2048), **rp.DEFAULT_REMOVESTARS)
            except Exception as e:   # noqa: BLE001
                assert type(g) is type(e) and str(g) == str(e)
                continue
            assert g.dtype == np.int32 and np.array_equal(g, ref)


def test_fitsio_lite_lazy_header_and_column_reader(tmp_path):
    """Header values are parsed on first access (same values as an eager parse, whatever the access path), and
    read_columns returns exactly the columns fitsio-style ``read`` returns, native-endian."""
    img = np.zeros((8, 12), np.float32)
    p = str(tmp_path / "a.fits")
    fitsio_lite.write_image(p, img, dict(synth.DEFAULT_HEADER))
    h = fitsio_lite.read_header(p)
    eager = {k: fitsio_lite._parse_value(dict.__getitem__(h, k)) if k in h._raw else dict.__getitem__(h, k) for k in list(h.keys())}
    assert h.get("NOSUCHKEY", 7) == 7 and "TAI" in h and "NOSUCHKEY" not in h
    assert h.get("CRPIX1") == eager["CRPIX1"] and isinstance(h["NAXIS1"], int) and h["SIMPLE"] is True
    assert dict(h.items()) == eager and h == eager and h.copy() == eager and list(h.values()) == list(eager.values())
    h["TAI"] = 1.5                                   # assignment of a real value is not re-parsed
    assert h["TAI"] == 1.5
    with pytest.raises(KeyError):
        h["NOSUCHKEY"]
    _img, cat = synth.make_case("sparse", 6)
    q = str(tmp_path / "b.fits")
    fitsio_lite.write_bintable(q, cat)
    data = fitsio_lite.read(q)
    cols = fitsio_lite.read_columns(q, ("ROWC", "PSFMAG", "NOBSERVE"))
    assert set(cols) == {"ROWC", "PSFMAG", "NOBSERVE"}
    for k, v in cols.items():
        assert v.dtype.isnative and v.dtype == data[k].dtype and np.array_equal(v, data[k]), k
    with pytest.raises(KeyError):
        fitsio_lite.read_columns(q, ("ROWC", "NOSUCHCOLUMN"))
    with pytest.raises(ValueError):
        fitsio_lite.read_columns(p, ("ROWC",))      # an image HDU, not a table


def test_native_ingest_equals_python(tmp_path):
    """lfd_fits_load_frame / lfd_catalog_rects (host code of the C-ABI library, no GPU needed) against the Python
    readers they stand in for: same payload bytes, same header values, same rectangles for every filter; files that
    are not of the plain kind are declined (None) so that the driver falls back to the Python path."""
    from lfd_b200 import detecttrails as dtm
    kinds = {(flt, field): kind for field, kind in ((100, "sparse"), (101, "dense"), (102, "trail")) for flt in "ugriz"}
    tree = synth.write_sdss_tree(str(tmp_path), 2888, 1, [100, 101, 102], filters=tuple("ugriz"), kinds=kinds)
    lfd_b200.setup(tree["bosspath"], tree["photoobjpath"], tree["photoreduxpath"], str(tmp_path))
    H, W = synth.FRAME_H, synth.FRAME_W
    slot_n, slot_p = np.zeros((H, W), np.uint32), np.zeros((H, W), np.uint32)
    for field in (100, 101, 102):
        for flt in "ugriz":
            fpath = sdssfiles.filename("frame", run=2888, camcol=1, field=field, filter=flt)
            raw = _lib.fits_load_frame(fpath, slot_n)
            hdr = fitsio_lite.read_raw_image_into(fpath, slot_p)
            assert raw is not None and np.array_equal(slot_n, slot_p)
            for k in _lib.HEADER_KEYS:
                assert fitsio_lite._parse_value(raw[k]) == hdr[k], k
            assert dtm._results_prefix(2888, 1, flt, field, dtm._RawHeader(raw)) == dtm._results_prefix(2888, 1, flt, field, hdr)
            opath = sdssfiles.filename("photoObj", run=2888, camcol=1, field=field)
            got = _lib.catalog_rects(opath, flt, (H, W), **rp.DEFAULT_REMOVESTARS)
            ref = star_rects(lfd_b200.removestars.read_photoObj_arrays(opath), flt, (H, W), **rp.DEFAULT_REMOVESTARS)
            assert got is not None and got.dtype == np.int32 and np.array_equal(got, ref), (field, flt)
    # other parameter values (fractional defaults, tight caps) and another frame shape go through the same arithmetic
    opath = sdssfiles.filename("photoObj", run=2888, camcol=1, field=101)
    cat = lfd_b200.removestars.read_photoObj_arrays(opath)
    for pr in (dict(rp.DEFAULT_REMOVESTARS, defaultxy=20.7, maxxy=33.5, pixscale=0.25, magcount=1, maxmagdiff=1.5),
               dict(rp.DEFAULT_REMOVESTARS, filter_caps={k: 19.5 for k in "ugriz"}, maxxy=1000)):
        for shape in ((H, W), (700, 900)):
            assert np.array_equal(_lib.catalog_rects(opath, "i", shape, **pr), star_rects(cat, "i", shape, **pr))
    # declined: wrong slot shape, an image where a table is expected (and vice versa), a missing file, a NaN in the table
    assert _lib.fits_load_frame(fpath, np.zeros((H, W + 4), np.uint32)) is None
    assert _lib.fits_load_frame(opath, slot_n) is None
    assert _lib.catalog_rects(fpath, "r", (H, W), **rp.DEFAULT_REMOVESTARS) is None
    assert _lib.catalog_rects(str(tmp_path / "nosuch.fits"), "r", (H, W), **rp.DEFAULT_REMOVESTARS) is None
    bad = {k: np.array(v, copy=True) for k, v in cat.items()}
    bad["PETROTH90"] = bad["PETROTH90"].astype(np.float32); bad["PETROTH90"][5, 1] = np.inf
    q = str(tmp_path / "bad.fits")
    fitsio_lite.write_bintable(q, bad)
    assert _lib.catalog_rects(q, "r", (H, W), **rp.DEFAULT_REMOVESTARS) is None
    # the loader takes the native path by default and the Python path on request: same record either way
    fr = (2888, 1, "g", 101)
    a = dtm._load_one(fr, rp.DEFAULT_REMOVESTARS, slot_n)
    old = dtm.NATIVE_INGEST
    try:
        dtm.NATIVE_INGEST = False
        b = dtm._load_one(fr, rp.DEFAULT_REMOVESTARS, slot_p)
    finally:
        dtm.NATIVE_INGEST = old
    assert a[0] == b[0] == "staged" and np.array_equal(a[3], b[3]) and a[4] == b[4] and np.array_equal(slot_n, slot_p)
    # the batched native ingest (one call, a pool of C++ threads) == the per-frame readers, item by item; a missing
    # catalog or frame only fails its own item
    frames = [(2888, 1, flt, field) for field in (100, 101, 102) for flt in "ugriz"]
    fpaths = [sdssfiles.filename("frame", run=r, camcol=c, field=fd, filter=fl) for (r, c, fl, fd) in frames]
    cpaths = [sdssfiles.filename("photoObj", run=r, camcol=c, field=fd) for (r, c, fl, fd) in frames]
    fpaths[4] = str(tmp_path / "missing-frame.fits")
    cpaths[7] = str(tmp_path / "missing-cat.fits")
    staging = np.zeros((len(frames), H, W), np.uint32)
    ing = _lib.ingest_batch(staging, fpaths, cpaths, [fr[2] for fr in frames], nthreads=4, **rp.DEFAULT_REMOVESTARS)
    assert ing is not None
    for i, fr in enumerate(frames):
        assert (ing.status_frame[i] == 0) == (i != 4) and (ing.status_cat[i] == 0) == (i != 7)
        if i == 4 or i == 7:
            continue
        ref = dtm._load_one(fr, rp.DEFAULT_REMOVESTARS, slot_p)
        assert ref[0] == "staged" and np.array_equal(staging[i], slot_p)
        assert np.array_equal(ing.rects[i, :ing.n_rects[i]], ref[3])
        assert str(dtm._NativePrefix(fr, ing, i)) == ref[4]


def test_scaled_frames_take_the_decoded_path(tmp_path):
    """A frame header with the trivial BSCALE = 1 / BZERO = 0 cards is plain payload for both raw readers (the native
    ingest must not decline it); a non-trivial scaling makes both decline, so that the driver decodes on the host like
    fitsio.read does (detecttrails.py:113)."""
    from lfd_b200 import _lib, fitsio_lite
    H, W = 40, 64
    img = np.random.default_rng(3).normal(0, 1, (H, W)).astype(np.float32)
    hdr = dict(synth.DEFAULT_HEADER)
    triv = str(tmp_path / "triv.fits")
    fitsio_lite.write_image(triv, img, dict(hdr, BSCALE=1.0, BZERO=0.0))
    scaled = str(tmp_path / "scaled.fits")
    fitsio_lite.write_image(scaled, img, dict(hdr, BSCALE=2.0, BZERO=0.5))
    want = img.astype(">f4").view(np.uint32)
    slot = np.zeros((H, W), np.uint32)
    raw = _lib.fits_load_frame(triv, slot)
    assert raw is not None and np.array_equal(slot, want)
    slot2 = np.zeros((H, W), np.uint32)
    fitsio_lite.read_raw_image_into(triv, slot2)
    assert np.array_equal(slot2, want) and np.array_equal(fitsio_lite.read_raw_image(triv)[0], want)
    assert _lib.fits_load_frame(scaled, slot) is None
    with pytest.raises(ValueError):
        fitsio_lite.read_raw_image(scaled)
    with pytest.raises(ValueError):
        fitsio_lite.read_raw_image_into(scaled, slot2)
    assert np.allclose(fitsio_lite.read(scaled), img * 2.0 + 0.5)
    # a header that claims more data than the image (PCOUNT) must not overrun the caller's slot
    big = str(tmp_path / "pcount.fits")
    fitsio_lite.write_image(big, img, dict(hdr, PCOUNT=4096, GCOUNT=1))
    guard = np.zeros((H + 8, W), np.uint32)
    assert _lib.fits_load_frame(big, guard[:H]) is None and not guard[H:].any()


def test_native_mapped_payload_copy(tmp_path):
    """The native reader copies a full-size frame payload from the mapped file with non-temporal stores: the same bytes
    as the Python reader, also into a slot that is not 32-byte aligned; a file shorter than its header claims is
    declined instead of faulting on the mapping."""
    tree = synth.write_sdss_tree(str(tmp_path), 2888, 1, [100], filters=("r",))
    lfd_b200.setup(tree["bosspath"], tree["photoobjpath"], tree["photoreduxpath"], str(tmp_path))
    H, W = synth.FRAME_H, synth.FRAME_W
    fpath = sdssfiles.filename("frame", run=2888, camcol=1, field=100, filter="r")
    ref = np.zeros((H, W), np.uint32)
    assert fitsio_lite.read_raw_image_into(fpath, ref) is not None
    slot = np.zeros((H, W), np.uint32)
    assert _lib.fits_load_frame(fpath, slot) is not None and np.array_equal(slot, ref)
    odd = np.zeros(H * W + 8, np.uint32)[3:3 + H * W].reshape(H, W)             # 12 bytes past the allocation's alignment
    assert _lib.fits_load_frame(fpath, odd) is not None and np.array_equal(odd, ref)
    short = str(tmp_path / "short.fits")
    data = open(fpath, "rb").read()
    open(short, "wb").write(data[:len(data) - 2880 * 3])
    assert _lib.fits_load_frame(short, slot) is None
