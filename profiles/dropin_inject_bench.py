"""Cost of injections in a drop-in run: DetectTrails(run, camcol, filter, injections=...).process() on a synthetic tree
of uncompressed FITS frames (the native ingest path), at batch 16 and 64, with K = 0, 1, 2, 4, 8 injections of one
Gaussian trail per frame (K = 0: no ``injections`` argument, the path of a run without them).  The repetitions
alternate over K, per batch size, after warm-up runs on a fresh ring of handles.  Per run: wall time, frames/s, injections/s, and whether
results.txt equals the K = 0 run's, and where the driver's thread spent its injection time (SPLIT).  Then k_capture_bases alone on a handle of each batch size (big-endian slots,
as the drop-in leaves them): event time per capture and the bytes it moves over that time.  The GPU's name and power
limit are read in the same call.

    python profiles/dropin_inject_bench.py [--frames 1024] [--distinct 32] [--out FILE.jsonl]
"""
import argparse
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import lfd_b200  # noqa: E402
from lfd_b200 import _lib, synth  # noqa: E402
from lfd_b200 import detecttrails as dtm  # noqa: E402
from lfd_b200 import inject as inj  # noqa: E402

# where the driver's thread spends its time on injections (seconds, per run): capture + submit_injected (host staging and
# enqueue), wait_array after submit_injected (blocked on the injected step's detection), and the lines (matching and
# formatting); the wrappers cost about a microsecond per call
SPLIT = {"capture_submit_s": 0.0, "wait_injected_s": 0.0, "lines_s": 0.0}


def _timed(fn, key, after=None):
    def wrapped(*a, **k):
        t0 = time.perf_counter()
        try:
            return fn(*a, **k)
        finally:
            if after is None or after(a[0]):
                SPLIT[key] += time.perf_counter() - t0
    return wrapped


_submit_injected, _wait_array = _lib.Handle.submit_injected, _lib.Handle.wait_array


def _submit_injected_marked(self, *a, **k):
    self._injected_step = True
    return _submit_injected(self, *a, **k)


def _wait_after_injected(h):
    was, h._injected_step = getattr(h, "_injected_step", False), False
    return was


_lib.Handle.capture_bases = _timed(_lib.Handle.capture_bases, "capture_submit_s")
_lib.Handle.submit_injected = _timed(_submit_injected_marked, "capture_submit_s")
_lib.Handle.wait_array = _timed(_wait_array, "wait_injected_s", after=_wait_after_injected)
inj.format_injection = _timed(inj.format_injection, "lines_s")
inj._recovered = _timed(inj._recovered, "lines_s")


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True)
    except OSError:
        return "unknown"
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def make_injections(k):
    def injections(frame, shape):
        h, w = shape
        rng = np.random.default_rng(synth.frame_seed(*frame) ^ 0xbe7c)
        out = []
        for _ in range(k):
            a = rng.uniform(0, np.pi)
            cx, cy, L = rng.uniform(0.25 * w, 0.75 * w), rng.uniform(0.25 * h, 0.75 * h), rng.uniform(300, 2000)
            out.append([{"p0": (cx - L / 2 * np.cos(a), cy - L / 2 * np.sin(a)), "p1": (cx + L / 2 * np.cos(a), cy + L / 2 * np.sin(a)),
                         "sigma": rng.uniform(0.8, 4.0), "peak": float(np.exp(rng.uniform(np.log(0.3), np.log(20.0))))}])
        return out
    return injections


def capture_times(batch, reps=20):
    """k_capture_bases event times (ms) on a handle of `batch` slots holding a big-endian batch."""
    h = _lib.Handle(synth.FRAME_H, synth.FRAME_W, max_batch=batch)
    try:
        p = lfd_b200.default_params()
        h.set_params(p[0], p[1])
        payload = np.repeat(synth.make_case("sparse", 5)[0][None], batch, axis=0).byteswap()
        h.submit(payload, None, flags=_lib.INPUT_BIGENDIAN)
        h.wait()
        ms = []
        for _ in range(reps):
            h.capture_bases()
            h.submit_injected([0])
            h.wait()
            ms.append([t[2] for t in h.kernel_times() if t[0] == "k_capture_bases"][0])
            h.submit(payload, None, flags=_lib.INPUT_BIGENDIAN)
            h.wait()
        return ms
    finally:
        h.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1024)
    ap.add_argument("--distinct", type=int, default=32)
    ap.add_argument("--batches", default="16,64")
    ap.add_argument("--ks", default="0,1,2,4,8")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    batches = [int(v) for v in a.batches.split(",")]
    ks = [int(v) for v in a.ks.split(",")]
    out_f = open(a.out, "a") if a.out else None

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        if out_f:
            out_f.write(line + "\n")
            out_f.flush()

    emit({"gpu": gpu_info(), "frames": a.frames, "distinct": a.distinct})
    root = tempfile.mkdtemp(prefix="lfd_b200_injbench_")
    try:
        # `distinct` fields generated, hard-linked up to `frames` names (as bench.py's drop-in leg)
        synth.write_sdss_tree(root, 2888, 1, range(100, 100 + a.distinct), filters=("r",), startfield=100, endfield=100 + a.frames)
        boss = os.path.join(root, "boss")
        fdir = os.path.join(boss, "photoObj", "frames", "301", "2888", "1")
        odir = os.path.join(boss, "photoObj", "301", "2888", "1")
        for k in range(a.distinct, a.frames):
            src = 100 + k % a.distinct
            os.link(os.path.join(fdir, "frame-r-002888-1-%04d.fits" % src), os.path.join(fdir, "frame-r-002888-1-%04d.fits" % (100 + k)))
            os.link(os.path.join(odir, "photoObj-002888-1-%04d.fits" % src), os.path.join(odir, "photoObj-002888-1-%04d.fits" % (100 + k)))
        lfd_b200.setup(boss, os.path.join(boss, "photoObj"), os.path.join(boss, "photo", "redux"), root)
        n_run = [0]

        def run(batch, k):
            out = os.path.join(root, "out%d" % n_run[0])
            n_run[0] += 1
            os.makedirs(out)
            kw = {"injections": make_injections(k)} if k else {}
            for key in SPLIT:
                SPLIT[key] = 0.0
            dt = lfd_b200.DetectTrails(run=2888, camcol=1, filter="r", savepath=out, batch=batch, **kw)
            t0 = time.perf_counter()
            dt.process()
            el = time.perf_counter() - t0
            res = open(os.path.join(out, "results.txt"), "rb").read()
            ninj = open(os.path.join(out, "injections.txt")).read().count("\n") if k else 0
            kt = {}
            for key, hs in dtm._handles.items():
                if key[0] == (synth.FRAME_H, synth.FRAME_W) and key[2] != "worst-case":
                    for h in hs:
                        for name, _p, ms, nl in h.kernel_times():
                            if name in ("k_capture_bases", "k_inject"):
                                kt.setdefault(name, []).append(ms)
            shutil.rmtree(out)
            return el, hashlib.sha256(res).hexdigest(), res.count(b"\n"), ninj, kt, {k_: round(v, 4) for k_, v in SPLIT.items()}

        ref = {}
        for batch in batches:
            # a fresh ring of handles with `batch` slots, as a run of its own would have; warm-up runs read the tree into
            # the page cache, create the handles and their injection bases
            for hs in dtm._handles.values():
                for h in hs:
                    h.close()
            dtm._handles.clear()
            run(batch, 0)
            run(batch, 1)
            for rep in range(a.reps):
                for k in ks:
                    el, digest, nl, ninj, kt, split = run(batch, k)
                    ref.setdefault(batch, digest)
                    emit({"rep": rep, "batch": batch, "K": k, "wall_s": round(el, 4), "frames_per_s": round(a.frames / el, 1),
                          "injections": ninj, "injections_per_s": round(ninj / el, 1), "detections": nl,
                          "results_equal_K0": digest == ref[batch],
                          "last_batch_kernel_ms": {n: [round(v, 4) for v in vs] for n, vs in kt.items()},
                          "driver_thread_split": split})
        for batch in batches:
            ms = capture_times(batch)
            nbytes = 2 * batch * synth.FRAME_H * synth.FRAME_W * 4
            med = float(np.median(ms))
            emit({"capture_batch": batch, "k_capture_bases_ms_median": round(med, 4), "ms_min": round(min(ms), 4),
                  "ms_max": round(max(ms), 4), "bytes": nbytes, "GB_per_s_at_median": round(nbytes / med / 1e6, 1)})
    finally:
        shutil.rmtree(root, ignore_errors=True)
        if out_f:
            out_f.close()


if __name__ == "__main__":
    main()
