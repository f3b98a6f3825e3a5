"""Drop-in for ``lfd.detecttrails.detecttrails``: ``DetectTrails`` and ``process_field``.

Mirrors /root/reference/lfd/detecttrails/detecttrails.py: constructor kwargs and defaults (:199-267,
including the quirk that ``params_dim=`` / ``params_removestars=`` kwargs land in ``params_bright``,
:253-256), frame-set selection ``_load`` (:290-342), loop order and ranges of ``process`` (:344-407,
``run-camcol`` strides fields by 50, ``endfield`` excluded), the results line (:115-117,127,131 - seven
of its brace groups are literal text in the reference and stay literal here), per-frame error capture
into errors.txt (:133-139) and the bz2 unpack path (:81-111).

What differs is where the work runs: frames are decoded on the host, grouped into batches, copied with
pinned cudaMemcpyAsync and pushed through liblfd_b200.so (one handle per GPU); results come back as one
small struct per frame and are written in the reference's frame order.
"""
import bz2
import os
import traceback

import numpy as _np

from . import _lib, inject as _inject, sdssfiles as files
from .processfield import result_from_device, setup_debug
from .removestars import read_photoObj_arrays, star_rects

try:
    import fitsio
except ImportError:  # pragma: no cover - depends on the image
    from . import fitsio_lite as fitsio

# cv2 enum values the reference re-exports (detecttrails.py:14-18); cv2 itself is not needed here
RETR_EXTERNAL, RETR_LIST, RETR_CCOMP, RETR_TREE = 0, 1, 2, 3
CHAIN_APPROX_NONE, CHAIN_APPROX_SIMPLE, CHAIN_APPROX_TC89_L1, CHAIN_APPROX_TC89_KCOS = 1, 2, 3, 4

__all__ = ["DetectTrails", "process_field", "process_fields", "default_params"]


def default_params():
    """The three default dicts of detecttrails.py:202-239."""
    params_bright = {
        "lwTresh": 5, "thetaTresh": 0.15, "dilateKernel": _np.ones((4, 4), _np.uint8),
        "contoursMode": RETR_LIST, "contoursMethod": CHAIN_APPROX_NONE, "minAreaRectMinLen": 1,
        "houghMethod": 20, "nlinesInSet": 3, "lineSetTresh": 0.15, "dro": 25, "debug": False}
    params_dim = {
        "minFlux": 0.02, "addFlux": 0.5, "lwTresh": 5, "thetaTresh": 0.15,
        "erodeKernel": _np.ones((3, 3), _np.uint8), "dilateKernel": _np.ones((9, 9), _np.uint8),
        "contoursMode": RETR_LIST, "contoursMethod": CHAIN_APPROX_NONE, "minAreaRectMinLen": 1,
        "houghMethod": 20, "nlinesInSet": 3, "lineSetTresh": 0.15, "dro": 20, "debug": False}
    params_removestars = {
        "pixscale": 0.396, "defaultxy": 20, "maxxy": 60,
        "filter_caps": {"u": 22.0, "g": 22.2, "r": 22.2, "i": 21.3, "z": 20.5},
        "magcount": 3, "maxmagdiff": 3, "debug": False}
    return params_bright, params_dim, params_removestars


# Opt-in (SURVEY.md 8(f) N2): write the seven header values instead of the reference's literal "{h['CRPIX2']}" ...
# placeholders, so that lfd.results.utils.parse_result_row (results/utils.py:185-210) can ingest the file.
# Default False = byte-identical to the reference.
FORMAT_HEADER_VALUES = False


def _load_frame(run, camcol, filter, field, raw=False):
    """detecttrails.py:73-117: resolve the path, unpack .bz2 if needed, read image + header.
    Returns (img, header_prefix_of_the_results_line[, big_endian]).  With raw=True and the built-in FITS reader the
    image is the undecoded big-endian payload (uint32 view) and big_endian is True: the device byte-swaps.

    A compressed frame is decompressed in memory with the built-in reader (no FITS_DUMP round trip through the file
    system: the reference writes the decompressed file, reads it and deletes it, detecttrails.py:90-111 - the pixels and
    header are the same); with the real ``fitsio`` module, which reads from paths only, the reference's temporary file
    is kept."""
    origfitspath = files.filename("frame", run=run, camcol=camcol, field=field, filter=filter)
    if not os.path.exists(origfitspath):
        bzpath = origfitspath + ".bz2"
        if not os.path.exists(bzpath):
            errmsg = ("File {0} or its bz2 compressed version not found. Are you sure they exist?")
            raise FileNotFoundError(errmsg.format(origfitspath))
        with open(bzpath, "rb") as compressedfits:
            fitsdata = bz2.decompress(compressedfits.read())          # releases the GIL: loader threads decompress in parallel
        if hasattr(fitsio, "read_image_bytes"):
            img, h, big_endian = fitsio.read_image_bytes(fitsdata)
            if not raw and big_endian:
                img, big_endian = img.view(">f4").astype(_np.float32), False
        else:
            try:
                fitsdmp = os.environ["FITS_DUMP"]
            except KeyError:
                fitsdmp = os.path.join(os.path.split(__file__)[0], "fits_dump/")
                os.makedirs(fitsdmp, exist_ok=True)
            fitspath = os.path.join(fitsdmp, os.path.split(origfitspath)[-1])
            with open(fitspath, "wb") as decompressed:
                decompressed.write(fitsdata)
            try:
                img, h, big_endian = fitsio.read(fitspath), fitsio.read_header(fitspath), False
            finally:
                os.remove(fitspath)
    else:
        big_endian = False
        if raw and hasattr(fitsio, "read_raw_image"):
            try:
                img, h = fitsio.read_raw_image(origfitspath)
                big_endian = True
            except ValueError:           # not a plain unscaled BITPIX=-32 image: decode on the host
                img = fitsio.read(origfitspath)
                h = fitsio.read_header(origfitspath)
        else:
            img = fitsio.read(origfitspath)
            h = fitsio.read_header(origfitspath)
    if not big_endian and img.dtype != _np.float32:
        img = img.astype(_np.float32)
    printit = _results_prefix(run, camcol, filter, field, h)
    return (img, printit, big_endian) if raw else (img, printit)


def _error_text(run, camcol, filter, field, exc):
    """The text detecttrails.py:133-139 appends to errors.txt for one failed frame."""
    return (f"{run} {camcol} {filter} {field}\n" +
            "".join(traceback.format_exception(type(exc), exc, exc.__traceback__, limit=3)) + str(exc) + "\n\n")


def _results_prefix(run, camcol, filter, field, h):
    """The header part of the results line (detecttrails.py:115-117); only the first fragment is an f-string in the
    reference, the seven other brace groups are literal text and stay literal unless FORMAT_HEADER_VALUES is set."""
    if FORMAT_HEADER_VALUES:
        return (f"{run} {camcol} {filter} {field} {h['TAI']} {h['CRPIX1']} "
                f"{h['CRPIX2']} {h['CRVAL1']} {h['CRVAL2']} {h['CD1_1']} "
                f"{h['CD1_2']} {h['CD2_1']} {h['CD2_2']} ")
    return (f"{run} {camcol} {filter} {field} {h['TAI']} {h['CRPIX1']} "
            "{h['CRPIX2']} {h['CRVAL1']} {h['CRVAL2']} {h['CD1_1']} "
            "{h['CD1_2']} {h['CD2_1']} {h['CD2_2']} ")


# FITS frames and photoObj tables are read by the library's host-side ingest (csrc/host_ingest.cuh) when they have the
# plain layout of the SDSS files; LFD_NATIVE_INGEST=0 keeps everything on the Python readers (same results, tested)
NATIVE_INGEST = os.environ.get("LFD_NATIVE_INGEST", "1") != "0"


class _RawHeader:
    """The nine header cards of the results line as returned by the native ingest, parsed on access like a
    FITSHeader (fitsio_lite._parse_value: same value formatting in the results line)."""

    def __init__(self, raw):
        self._raw = raw

    def __getitem__(self, key):
        from .fitsio_lite import _parse_value
        return _parse_value(self._raw[key])


class _NativePrefix:
    """Results-line prefix of a natively ingested frame, formatted only if the frame turns out to be a detection."""
    __slots__ = ("frame", "ing", "j")

    def __init__(self, frame, ing, j):
        self.frame, self.ing, self.j = frame, ing, j

    def __str__(self):
        return _results_prefix(*self.frame, _RawHeader(self.ing.header(self.j)))


def _stage(slot, img, big_endian):
    """Put a frame into a pinned staging slot (viewed as uint32) as raw big-endian float32 payload."""
    if big_endian:
        slot[...] = img
    else:
        slot[...] = _np.ascontiguousarray(img, _np.float32).astype(">f4").view(_np.uint32)


def _load_one(frame, params_removestars, slot=None, want_rects=True):
    """Host side of one frame through the general (Python) readers - compressed frames, other layouts, anything the
    native batch ingest declined: FITS image + header line prefix, photoObj catalog -> blot rectangles.  With ``slot``
    (a row of a handle's pinned staging viewed as uint32) a frame of that shape is left there as raw big-endian payload.
    Returns ("staged", None, True, rects, printit) | ("ok", pixels, big_endian, rects, printit) | ("err", exc)."""
    run, camcol, filter, field = frame
    try:
        img, printit, big_endian = _load_frame(run, camcol, filter, field, raw=True)
        opath = files.filename("photoObj", run=run, camcol=camcol, field=field)
        rects = _lib.catalog_rects(opath, filter, img.shape, **dict(params_removestars)) if NATIVE_INGEST else None
        if rects is None:                                    # not the plain table layout, or a value the reference raises on
            cat = read_photoObj_arrays(opath)
            rects = star_rects(cat, filter, img.shape, **dict(params_removestars))
        if slot is not None and tuple(img.shape) == tuple(slot.shape):
            _stage(slot, img, big_endian)
            return ("staged", None, True, rects, printit)
        return ("ok", img, big_endian, rects, printit)
    except Exception as e:   # noqa: BLE001 - the reference swallows everything per frame
        return ("err", e)


_handles = {}
N_RING = 3      # handles per frame shape: one computing, one submitted (crossing PCIe), one being filled by the loaders


def _handle_caps():
    """Optional capacities of the ring handles (tests shrink them to exercise the overflow retry)."""
    return (int(os.environ.get("LFD_MAX_RUNS", 0)), int(os.environ.get("LFD_MAX_COMPONENTS", 0)))


def _batch_handles(shape, batch, device, count=N_RING):
    key = (shape, device, _handle_caps())
    hs = _handles.get(key)
    if hs is None or hs[0].B < batch or len(hs) < count:
        for h in hs or []:
            h.close()
        mr, mc = _handle_caps()
        hs = [_lib.Handle(shape[0], shape[1], max_batch=batch, device=device, max_runs=mr, max_components=mc) for _ in range(count)]
        if "LOCAL_RANK" in os.environ:                 # torchrun: share the bridge's copy slots with the neighbouring ranks
            from .sharding import apply_h2d_gate
            apply_h2d_gate(hs, device)
        _handles[key] = hs
    return hs


def _big_handle(shape, device):
    """One-frame handle with worst-case run / contour capacities: a frame that overflowed the batch handles' work lists
    is run again here, so it gets the result the reference gives instead of an errors.txt entry."""
    key = (shape, device, "worst-case")
    h = _handles.get(key)
    if h is None:
        worst = shape[0] * ((shape[1] + 1) // 2)
        h = _handles[key] = [_lib.Handle(shape[0], shape[1], max_batch=1, device=device, max_runs=worst, max_components=worst)]
    return h[0]


def _probe_shape(frames, params_removestars):
    """Shape of the first frame that can be read (SDSS frames of a run all have one shape), compressed ones included;
    None if none of the first few can be read."""
    for fr in frames[:8]:
        try:
            run, camcol, filter, field = fr
            path = files.filename("frame", run=run, camcol=camcol, field=field, filter=filter)
            if os.path.exists(path):
                h = fitsio.read_header(path)
                return (int(h["NAXIS2"]), int(h["NAXIS1"]))
            img, _p, _b = _load_frame(run, camcol, filter, field, raw=True)
            return tuple(int(v) for v in img.shape)
        except Exception:   # noqa: BLE001
            continue
    return None


def _decode_batch(h, shape, n):
    """lfd_wait + the verdict of every frame of the batch: [("ok", detected, result dict | None) | ("err", exc) |
    ("overflow",)].  Only frames with a rectangle detection or a status bit go through the per-frame decoder."""
    arr = h.wait_array()
    out = [("ok", False, None)] * n
    busy = _np.nonzero((arr["status"] != 0) | (arr["rect_detection"] == 1).any(axis=1))[0]
    for k in busy:
        k = int(k)
        r = h._results[k]
        if r.status & _lib.FRAME_OVERFLOW:
            out[k] = ("overflow",)
            continue
        try:
            det, res = False, None
            for p in (0, 1):
                if r.rect_detection[p] >= 0:
                    det, res = result_from_device(r, p, shape)
                    if det:
                        break
            out[k] = ("ok", det, res)
        except Exception as e:   # noqa: BLE001
            out[k] = ("err", e)
    return out


def compute_fields_iter(frames, params_bright, params_dim, params_removestars, batch=16, device=0, loaders=None,
                        injections=None, injection_tables=None):
    """Run an ordered list of (run, camcol, filter, field) through the GPU in batches.  Generator: yields, batch by batch
    and in list order, ``(index of the batch's first frame, records)`` with one record per frame - ("line", results_line)
    for a detection, ("none", "") for no detection, ("err", errors_text) for a failure - exactly what the reference's
    per-frame loop would append.

    Pipeline (three handles of the common frame shape form a ring): while batch k-1 computes and batch k crosses PCIe,
    ONE native call (lfd_ingest_batch, a pool of C++ threads, GIL released) reads the raw big-endian FITS payloads of
    batch k+1 straight into the third handle's pinned staging and filters its photoObj catalogs; the first kernel
    byte-swaps.  Frames the native reader declines (compressed, scaled, another BITPIX) go through the Python readers on
    loader threads (bz2 releases the GIL) and end up in the same staging slots; frames of another shape use a cached
    handle of their own.  A frame whose run / contour lists overflow the batch handles is re-run on a worst-case-capacity
    handle instead of being reported as an error.

    With ``injections`` (see DetectTrails) the record of every frame with a verdict carries a third item, the frame's
    lines of the injection table: after a batch is collected, its handle makes the frames still in its slots the
    injection bases (lfd_capture_bases, a device copy) and runs each injection on the slot of its frame, in steps of
    the handle's slots.  ``injection_tables`` is the pool their ``profile`` / ``lightcurve`` keys index.  The
    injections of a batch are checked when it is loaded, before it is submitted: a bad one raises ValueError."""
    from concurrent.futures import ThreadPoolExecutor
    frames = list(frames)
    debug = bool(params_bright["debug"] or params_dim["debug"])
    if debug and injections is not None:
        raise ValueError("injections are not supported with debug=True (the debug path runs frames one at a time on the host)")
    if debug:
        recs = _compute_fields_debug(frames, params_bright, params_dim, params_removestars)
        for i0 in range(0, len(frames), max(int(batch), 1)):
            yield i0, recs[i0:i0 + max(int(batch), 1)]
        return
    batch = max(int(batch), 1)
    chunks = [frames[i:i + batch] for i in range(0, len(frames), batch)]
    pr = dict(params_removestars)
    shape0 = _probe_shape(frames, pr)
    ring = []
    if shape0 is not None:
        try:
            ring = _batch_handles(shape0, batch, device)
        except Exception:   # noqa: BLE001 - reported per frame below, when the submit fails the same way
            ring = []
    nload = (loaders or int(os.environ.get("LFD_LOADER_THREADS", 0)) or max(2, min(12, (os.cpu_count() or 2))))

    def load_chunk(ci, fpool):
        """Loader job of one batch (worker thread): native ingest of the whole batch, Python readers for the rest."""
        chunk = chunks[ci]
        h = ring[ci % len(ring)] if ring else None
        st = h.host_frames.view(_np.uint32) if h is not None else None
        items = [None] * len(chunk)
        ing = None
        if h is not None and NATIVE_INGEST:
            try:
                fpaths = [files.filename("frame", run=r, camcol=c, field=fd, filter=fl) for (r, c, fl, fd) in chunk]
                cpaths = [files.filename("photoObj", run=r, camcol=c, field=fd) for (r, c, fl, fd) in chunk]
                ing = _lib.ingest_batch(st, fpaths, cpaths, [fr[2] for fr in chunk], nthreads=nload, **pr)
            except Exception:   # noqa: BLE001 - e.g. a filter that is not one of ugriz: the per-frame path raises it properly
                ing = None
        rest = []
        for j, fr in enumerate(chunk):
            if ing is not None and ing.status_frame[j] == 0 and ing.status_cat[j] == 0:
                items[j] = ("staged", None, True, ing.rects[j, :ing.n_rects[j]], _NativePrefix(fr, ing, j))
            else:
                rest.append(j)
        if rest:
            for j, it in zip(rest, fpool.map(lambda jj: _load_one(chunk[jj], pr, st[jj] if st is not None else None), rest)):
                items[j] = it
        return items

    def finish(entry):
        """Collect one submitted batch -> {global index: ("ok", det, res) | ("err", exc)}."""
        if entry[0] == "failed":
            return {g: ("err", entry[2]) for g in entry[1]}
        _tag, h, shape, gidx, rects, big_endian = entry
        try:
            dec = _decode_batch(h, shape, len(gidx))
        except Exception as e:   # noqa: BLE001
            return {g: ("err", e) for g in gidx}
        out = {}
        for k, g in enumerate(gidx):
            d = dec[k]
            if d[0] == "overflow":
                try:
                    big = _big_handle(shape, device)
                    big.set_params(params_bright, params_dim)
                    if big_endian:
                        big.host_frames.view(_np.uint32)[0] = h.host_frames.view(_np.uint32)[k]
                    else:
                        big.host_frames[0] = h.host_frames[k]
                    big.submit(1, [rects[k]], flags=_lib.INPUT_BIGENDIAN if big_endian else 0)
                    d = _decode_batch(big, shape, 1)[0]
                    if d[0] == "overflow":
                        d = ("err", _lib.LfdError(_lib.LFD_E_CAPACITY, "per-frame work list overflow"))
                except Exception as e:   # noqa: BLE001
                    d = ("err", e)
            out[g] = d
        return out

    def submit(h, shape, gidx, rects, big_endian):
        try:
            h.set_params(params_bright, params_dim)
            h.submit(len(gidx), rects, flags=_lib.INPUT_BIGENDIAN if big_endian else 0)
            return ("entry", h, shape, gidx, rects, big_endian)
        except Exception as e:   # noqa: BLE001
            return ("failed", gidx, e)

    hough = (float(params_bright["houghMethod"]), float(params_dim["houghMethod"]))
    injection_tables = list(injection_tables) if injection_tables else None
    ntab = len(injection_tables) if injection_tables else 0
    tables_set = set()          # id() of the handles that hold this call's table pool

    def specs_of(ci, items):
        """{global index: checked injections} of the frames of batch ci that were read (their shape is known)."""
        specs = {}
        if injections is not None:
            for j, it in enumerate(items):
                if it[0] != "err":
                    shp = shape0 if it[0] == "staged" else tuple(int(v) for v in it[1].shape)
                    specs[ci * batch + j] = _inject.check_injections(injections(chunks[ci][j], shp), ntab)
        return specs

    def inject(entry, outcome, specs):
        """Run the injections of a collected batch from the frames still in its handle's slots (slot k holds gidx[k]);
        each frame with a verdict gets its injection lines appended to its outcome.  An injected frame that overflows
        is reported in its status, not retried."""
        if entry[0] != "entry":
            return
        _tag, h, shape, gidx, _rects, _be = entry
        jobs = [(slot, g, k, ts) for slot, g in enumerate(gidx) if outcome.get(g, ("err",))[0] == "ok"
                for k, ts in enumerate(specs.get(g, ()))]
        if not jobs:
            return
        if injection_tables and id(h) not in tables_set:
            h.set_trail_tables(injection_tables)
            tables_set.add(id(h))
        h.capture_bases()
        rows = {}
        for i in range(0, len(jobs), h.B):
            step = jobs[i:i + h.B]
            h.submit_injected([j[0] for j in step], [j[3] for j in step])
            for (_slot, g, k, ts), r in zip(step, h.wait_array()):
                rows.setdefault(g, []).append(_inject.format_injection(frames[g], k, outcome[g][1], ts, r,
                                                                      _inject._recovered(r, ts, shape, hough)))
        for g, lines in rows.items():
            outcome[g] = outcome[g] + ("".join(lines),)

    def records_of(ci, items, outcome):
        recs = []
        base = ci * batch
        for j, (run, camcol, filter, field) in enumerate(chunks[ci]):
            item, oc = items[j], outcome.get(base + j)
            exc = item[1] if item[0] == "err" else (oc[1] if oc is not None and oc[0] == "err" else None)
            if exc is None and oc is None:
                exc = _lib.LfdError(_lib.LFD_E_STATE, "frame was not processed")
            if exc is not None:
                recs.append(("err", _error_text(run, camcol, filter, field, exc)))
            elif oc[1]:
                res = oc[2]
                recs.append(("line", str(item[4]) + f"{res['x1']} {res['y1']} {res['x2']} {res['y2']}\n"))
            else:
                recs.append(("none", ""))
            if exc is None and len(oc) > 3:
                recs[-1] += (oc[3],)
        return recs

    with ThreadPoolExecutor(max_workers=2) as bpool, ThreadPoolExecutor(max_workers=nload) as fpool:
        futs = {0: bpool.submit(load_chunk, 0, fpool)} if chunks else {}
        inflight = []            # [(ci, items, submitted entries, {outcomes known so far}, injections)] in submission order
        collected = []           # the same for collected batches whose injections and records are still to come

        def collect(upto):
            """Collect every submitted batch with index <= upto, oldest first: verdicts and the overflow retry, which
            reads the handle's host staging before the next load overwrites it."""
            while inflight and inflight[0][0] <= upto:
                b = inflight.pop(0)
                for e in b[2]:
                    b[3].update(finish(e))
                collected.append(b)

        def release():
            """Run the injections of the collected batches and yield their records.  The injections use only the
            device slots and the library's own staging, so they overlap the two loads in flight."""
            while collected:
                cj, itj, ents, oc, spj = collected.pop(0)
                for e in ents:
                    inject(e, oc, spj)
                yield cj * batch, records_of(cj, itj, oc)

        try:
            for ci, chunk in enumerate(chunks):
                # the handle batch ci+1 loads into is the one batch ci-2 used (ring of three): collect that one, then start
                # the next load so that it runs while batch ci is submitted and batch ci-1 computes.  Batch ci-2's
                # injections run while loads ci and ci+1 are in flight and before batch ci's frames are copied: the
                # injected steps' small host->device copies would otherwise queue behind that batch copy
                collect(ci - (len(ring) - 1 if ring else 1))
                if ci + 1 < len(chunks):
                    futs[ci + 1] = bpool.submit(load_chunk, ci + 1, fpool)
                yield from release()
                items = futs.pop(ci).result()
                specs = specs_of(ci, items)
                base = ci * batch
                h = ring[ci % len(ring)] if ring else None
                outcome = {}
                entries = []
                staged = [j for j, it in enumerate(items) if it[0] == "staged"]
                if staged:
                    # staged frames sit in their own slots; compact them to the front (a frame that failed or took
                    # another path leaves a hole)
                    st = h.host_frames.view(_np.uint32)
                    for k, j in enumerate(staged):
                        if k != j:
                            st[k] = st[j]
                    entries.append(submit(h, shape0, [base + j for j in staged], [items[j][3] for j in staged], True))
                others = {}
                for j, it in enumerate(items):
                    if it[0] == "ok":
                        others.setdefault((tuple(it[1].shape), bool(it[2])), []).append(j)
                for (shape, big_endian), idxs in others.items():
                    # another frame shape (or no ring): a cached handle of that shape, run to completion right away
                    gidx = [base + j for j in idxs]
                    ent = ("failed",)
                    try:
                        hh = _batch_handles(shape, batch, device, count=1)[0]
                        stg = hh.host_frames.view(_np.uint32) if big_endian else hh.host_frames
                        for slot, j in enumerate(idxs):
                            stg[slot] = items[j][1]
                        ent = submit(hh, shape, gidx, [items[j][3] for j in idxs], big_endian)
                        outcome.update(finish(ent))
                    except Exception as e:   # noqa: BLE001
                        outcome.update({g: ("err", e) for g in gidx})
                    inject(ent, outcome, specs)
                inflight.append((ci, items, entries, outcome, specs))
            collect(len(chunks))
            yield from release()
        finally:
            # the consumer stopped early (or something raised): collect what is still on the GPU, so that the cached
            # handles are not left with a pending batch ("previous batch not collected" on their next use)
            for _cj, _itj, ents, _oc, _sp in inflight + collected:
                for e in ents:
                    if e[0] == "entry":
                        try:
                            e[1].wait()
                        except Exception:   # noqa: BLE001
                            pass
            for fu in futs.values():
                try:
                    fu.result()                       # a loader still writing into a handle's staging
                except Exception:   # noqa: BLE001
                    pass


def compute_fields(frames, params_bright, params_dim, params_removestars, batch=16, device=0, loaders=None,
                   injections=None, injection_tables=None):
    """All records of ``compute_fields_iter`` as one list in frame order."""
    out = []
    for _i0, recs in compute_fields_iter(frames, params_bright, params_dim, params_removestars, batch=batch, device=device,
                                         loaders=loaders, injections=injections, injection_tables=injection_tables):
        out.extend(recs)
    return out


def _compute_fields_debug(frames, params_bright, params_dim, params_removestars):
    """debug=True: one frame at a time through the standalone stage functions, which write the reference's debug
    images into $DEBUG_PATH and print the check_theta values (detecttrails.py:119-131 literally)."""
    from .processfield import process_field_bright, process_field_dim
    from .removestars import remove_stars
    records = []
    for (run, camcol, filter, field) in frames:
        try:
            img, printit = _load_frame(run, camcol, filter, field)
            img = remove_stars(_np.ascontiguousarray(img, _np.float32), run, camcol, filter, field, **params_removestars)
            img = _np.ascontiguousarray(img[::-1])                   # cv2.flip(img, 0)
            detection, res = process_field_bright(img, **params_bright)
            if not detection:
                detection, res = process_field_dim(img, **params_dim)
            if detection:
                records.append(("line", printit + f"{res['x1']} {res['y1']} {res['x2']} {res['y2']}\n"))
            else:
                records.append(("none", ""))
        except Exception as e:   # noqa: BLE001
            traceback.print_exception(type(e), e, e.__traceback__, limit=3)
            records.append(("err", _error_text(run, camcol, filter, field, e)))
    return records


def write_records(results, errors, records):
    for rec in records:
        kind, text = rec[0], rec[1]
        if kind == "line":
            results.write(text)
        elif kind == "err":
            errors.write(text)


def _progress_key(frame):
    run, camcol, filter, field = frame
    return f"{run} {camcol} {filter} {field}"


def read_progress(path):
    """Frames already finished by an earlier, interrupted run (one "run camcol filter field status" line each)."""
    done = set()
    if path and os.path.exists(path):
        with open(path) as f:
            for line in f:
                t = line.split()
                if len(t) >= 5:
                    done.add(" ".join(t[:4]))
    return done


def process_fields(results, errors, frames, params_bright, params_dim, params_removestars, batch=16, device=0,
                   distributed=None, compute=None, progress=None, injections=None, injection_tables=None,
                   injection_results=None):
    """Process an ordered list of (run, camcol, filter, field); results/errors are written in list order,
    exactly the lines the reference's per-frame loop would write, and flushed after every GPU batch (the reference
    appends frame by frame, detecttrails.py:127-139: a killed run keeps what it finished).

    ``injections`` / ``injection_tables``: see DetectTrails; the injection lines a record carries as its third item go
    to the open file ``injection_results``, in frame order, written and flushed with the batch's results and errors.

    With ``torch.distributed`` initialised (one process per GPU, e.g. under torchrun) the list is sharded by
    frame across the ranks - blocks of ``batch`` consecutive frames dealt round-robin, no data-path collective -
    and rank 0 gathers the per-frame records and writes them in the original order (lfd_b200/sharding.py).
    ``distributed=False`` forces the single-process path; ``compute`` replaces the GPU stage (tests)."""
    from . import sharding
    frames = list(frames)
    if distributed is None:
        distributed = sharding.is_distributed()
    # resumable runs (SURVEY.md 8(f) N3): `progress` is a text file with one line per finished frame; frames listed
    # there are skipped, and the file is extended batch by batch, right after the batch's results/errors lines are flushed
    if progress:
        done = read_progress(progress)
        frames = [fr for fr in frames if _progress_key(fr) not in done]
    writer = (not distributed) or sharding.rank() == 0

    def emit(part, recs):
        write_records(results, errors, recs)
        results.flush(); errors.flush()
        if injection_results is not None:
            injection_results.write("".join(rec[2] for rec in recs if len(rec) > 2))
            injection_results.flush()
        if progress:
            with open(progress, "a") as pf:
                pf.write("".join(_progress_key(fr) + " " + rec[0] + "\n" for fr, rec in zip(part, recs)))

    if not distributed:
        if compute is not None:                       # injected compute stage (tests): one call per `batch * 32` frames
            step = max(batch, 1) * 32
            for i0 in range(0, len(frames), step):
                emit(frames[i0:i0 + step], compute(frames[i0:i0 + step]))
            return
        for i0, recs in compute_fields_iter(frames, params_bright, params_dim, params_removestars, batch=batch, device=device,
                                            injections=injections, injection_tables=injection_tables):
            emit(frames[i0:i0 + len(recs)], recs)
        return
    compute = compute or (lambda fr: compute_fields(fr, params_bright, params_dim, params_removestars, batch=batch, device=device,
                                                    injections=injections, injection_tables=injection_tables))
    # frames per gather: every rank runs `32` of its own batches between two gathers (the ring drains at a gather)
    chunk = max(batch, 1) * sharding.world_size() * 32
    for i0 in range(0, len(frames), chunk):
        part = frames[i0:i0 + chunk]
        recs = sharding.run_sharded(part, compute, block=batch)
        if writer:
            emit(part, recs)


def process_field(results, errors, run, camcol, filter, field, params_bright, params_dim, params_removestars):
    """detecttrails.py:30-143 for one frame (always in this process: a single frame is never sharded)."""
    process_fields(results, errors, [(run, camcol, filter, field)], params_bright, params_dim,
                   params_removestars, batch=1, distributed=False)


class DetectTrails:
    """Convenience class that processes targeted SDSS frames (detecttrails.py:146-407).

    Extra, optional kwargs that the reference does not have: ``batch`` (frames per GPU batch, default 16),
    ``device`` (CUDA device index, default: LOCAL_RANK under torchrun, else 0) and ``resume`` (path of a progress
    file, or True for ``<savepath>/progress.txt``: frames listed there are skipped and finished frames are appended,
    so an interrupted run can be restarted without duplicating lines - the reference only appends, detecttrails.py:349).
    Under torchrun (torch.distributed initialised) the frame list is sharded over the ranks and rank 0 writes.

    Completeness of the run itself: ``injections``, a callable ``injections(frame, shape) -> [[trail, ...], ...]``
    called with ``frame`` = (run, camcol, filter, field) and the frame's (H, W) as read, returns the frame's injections,
    each a list of at most 16 trails in ``inject.recovery``'s format (``p0``, ``p1``, ``sigma``, ``peak``, optional
    ``profile`` / ``lightcurve`` indices into ``injection_tables``), end points in the un-flipped FITS orientation.
    Every frame with a verdict gets them, injected on the device into the copy of the frame already there (no second
    read or upload), and one line per injection goes to ``injection_results`` (default ``<savepath>/injections.txt``,
    appended like results.txt; inject.read_injections reads it): the frame, the index k of the injection, the
    frame's own verdict, the injected frame's verdict, line and ``recovered`` (inject.recovery's default tolerances),
    and the trails.  The callable must return the same injections for the same frame on every call (e.g. seeded
    from synth.frame_seed): sharded and resumed runs rely on it.  A bad injection (more than 16 trails, a value that
    is not finite, sigma <= 0 for a Gaussian, a table index outside the pool) raises ValueError before its batch is
    submitted; so does ``debug=True``.  results.txt, errors.txt and the progress file are the same as without."""

    def __init__(self, **kwargs):
        savepth = (kwargs["savepath"] if "savepath" in kwargs else ".")
        self.kwargs = kwargs
        self.params_bright, self.params_dim, self.params_removestars = default_params()
        self.batch = int(kwargs.get("batch", 16))
        if "device" in kwargs:
            self.device = int(kwargs["device"])
        else:                                          # under torchrun: LOCAL_RANK, spread over the node's GPUs (sharding.py)
            from .sharding import spread_device
            self.device = spread_device(os.environ.get("LOCAL_RANK", 0)) if "LOCAL_RANK" in os.environ else 0
        resume = kwargs.get("resume", None)
        self.progress = (os.path.join(savepth, "progress.txt") if resume is True else resume) or None
        self.injections = kwargs.get("injections", None)
        self.injection_tables = kwargs.get("injection_tables", None)
        self.injection_results = kwargs.get("injection_results", os.path.join(savepth, "injections.txt"))

        if "results" in kwargs:
            self.results = kwargs["results"]
        else:
            self.results = os.path.join(savepth, "results.txt")
        if "errors" in kwargs:
            self.errors = kwargs["errors"]
        else:
            self.errors = os.path.join(savepth, "errors.txt")

        # reference behaviour, kept on purpose: all three land in params_bright (detecttrails.py:251-256)
        if "params_bright" in kwargs:
            self.params_bright = kwargs["params_bright"]
        if "params_dim" in kwargs:
            self.params_bright = kwargs["params_dim"]
        if "params_removestars" in kwargs:
            self.params_bright = kwargs["params_removestars"]

        if "debug" in kwargs:
            self.debug = kwargs.pop("debug")
            self.params_bright["debug"] = self.debug
            self.params_dim["debug"] = self.debug
            self.params_removestars["debug"] = self.debug
        if any([self.params_removestars["debug"], self.params_bright["debug"], self.params_dim["debug"]]):
            setup_debug()

        self._load()

    def _runInfo(self):
        rl = files.runlist()
        w, = _np.where(rl["run"] == self._run)
        if len(w) == 0:
            raise ValueError("Run %s not found in runList.par" % self._run)
        return rl[w]["startfield"][0], rl[w]["endfield"][0]

    def _getRuns(self):
        rl = files.runlist()
        runs = rl["run"]
        if runs is None:
            raise ValueError("Unable to retrieve runs. Retrieved NoneType.")
        return runs

    def _load(self):
        """kwargs -> self._pick (detecttrails.py:290-342)."""
        self._run, self._camcol, self._field = int(0), int(0), int(0)
        self._filter, self._pick = str(0), str(0)
        kwargs = self.kwargs
        if "run" in kwargs:
            self._run = kwargs["run"]
            self._pick = "run"
        if "camcol" in kwargs:
            if kwargs["camcol"] not in (1, 2, 3, 4, 5, 6):
                raise ValueError("Nonexisting camcol")
            self._camcol = kwargs["camcol"]
            self._pick = "run-camcol"
        if "field" in kwargs or "frame" in kwargs:
            if self._camcol == 0:
                raise ValueError("send camcol= ")
            self._field = kwargs["field"] if "field" in kwargs else kwargs["frame"]
        if "filter" in kwargs:
            if kwargs["filter"] not in ("u", "g", "r", "i", "z"):
                raise ValueError("Nonexistting filter")
            self._filter = kwargs["filter"]
            if self._camcol != 0:
                self._pick = "camcol-filter"
            if self._run != 0:
                self._pick = "run-filter"
            if (self._camcol != 0) and (self._run != 0):
                self._pick = "run-camcol-filter"
        if "filter" not in kwargs:
            if (self._field != 0) and (self._camcol != 0):
                self._pick = "camcol-frame"
        if (self._field != 0) and (self._camcol != 0) and (self._filter != "0"):
            self._pick = "field"

    def frame_list(self):
        """The (run, camcol, filter, field) sequence ``process`` visits, in the reference's order."""
        out = []
        filters = ("u", "g", "r", "i", "z")
        camcols = (1, 2, 3, 4, 5, 6)
        if self._pick == "camcol-filter":
            for _run in self._getRuns():
                self._run = _run
                startfield, endfield = self._runInfo()
                out += [(_run, self._camcol, self._filter, f) for f in range(startfield, endfield, 1)]
            self._run = 0
        if self._pick == "run":
            startfield, endfield = self._runInfo()
            for c in camcols:
                for flt in filters:
                    out += [(self._run, c, flt, f) for f in range(startfield, endfield, 1)]
        if self._pick == "run-filter":
            startfield, endfield = self._runInfo()
            for c in camcols:
                out += [(self._run, c, self._filter, f) for f in range(startfield, endfield, 1)]
        if self._pick == "run-camcol":
            startfield, endfield = self._runInfo()
            for flt in filters:
                out += [(self._run, self._camcol, flt, f) for f in range(startfield, endfield, 50)]
        if self._pick == "run-camcol-filter":
            startfield, endfield = self._runInfo()
            out += [(self._run, self._camcol, self._filter, f) for f in range(startfield, endfield, 1)]
        if self._pick == "camcol-frame":
            out += [(self._run, self._camcol, flt, self._field) for flt in filters]
        if self._pick == "field":
            out.append((self._run, self._camcol, self._filter, self._field))
        return out

    def process(self):
        """Run the selected frames; results/errors (and injection) files are opened in append mode like the original."""
        import contextlib
        with open(self.results, "a") as results, open(self.errors, "a") as errors, \
                (open(self.injection_results, "a") if self.injections is not None else contextlib.nullcontext()) as inj:
            process_fields(results, errors, self.frame_list(), self.params_bright, self.params_dim,
                           self.params_removestars, batch=self.batch, device=self.device, progress=self.progress,
                           injections=self.injections, injection_tables=self.injection_tables, injection_results=inj)
