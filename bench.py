#!/usr/bin/env python
"""bench.py - frames/s of lfd.detecttrails' full per-frame detect on synthetic SDSS-shaped frames.

  python bench.py --gpus N --steps K --warmup W            (our arm; N>1 under torchrun, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K ...  (the reference's CPU path on the host cores)

A step = one batch of B frames (2048x1489 float32, config-3 mix of sparse / dense / trail / satellite
fields with star catalogs) through star mask -> flip -> bright -> dim-if-needed -> result.
`value` is measured with the batch already resident in HBM; `e2e` is the same metric through the C-ABI
with HOST (pinned) frames, host->device and device->host copies inside the timed region, two handles
double-buffered so copies overlap compute.  Frames are independent: ranks shard frames, no collective.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from lfd_b200 import synth  # noqa: E402

H, W = synth.FRAME_H, synth.FRAME_W
N = H * W
METRIC = "frames/sec (2048x1489 SDSS field, full detect)"
WORKLOADS = {"config3": "config3-camcol-mix", "config4": "config4-high-sensitivity-dim", "config5": "config5-hough-canny-microbench"}
WORKLOAD = WORKLOADS["config3"]


def workload_params(args):
    """(workload name, params_bright, params_dim) of BASELINE.json config 3 (the drop-in's defaults, detecttrails.py:202-239)
    or config 4 (high-sensitivity dim pass: 15x15 dilation kernel, houghMethod 1..5 = finer rho; theta is a literal in the
    reference, processfield.py:488-489)."""
    import lfd_b200
    pb, pd, _pr = lfd_b200.default_params()
    if args.workload == "config4":
        pd = dict(pd, dilateKernel=np.ones((15, 15), np.uint8), houghMethod=args.hough_method)
        return "%s(dilate15x15,houghMethod=%g)" % (WORKLOADS["config4"], args.hough_method), pb, pd
    return WORKLOADS["config3"], pb, pd


def env_int(k, d):
    return int(os.environ.get(k, d))


def dump_arrays(outdir, arrays):
    """--dump-outputs: every array as DIR/<name>.npy in float64 (integer results and float32 values convert exactly), so
    that two builds run with the same arguments (hence on the same seeded inputs) can be compared output for output."""
    os.makedirs(outdir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(outdir, name + ".npy"), np.asarray(a, np.float64))


def result_arrays(leg, raw_results):
    """The lfd_result structs a caller of lfd_wait receives for the frames of one step, one array per field, frames first."""
    from lfd_b200 import _lib
    rec = np.frombuffer(b"".join(raw_results), dtype=np.dtype(_lib.Result))
    return {"%s_%s" % (leg, f.rstrip("_")): rec[f] for f in rec.dtype.names}


def make_pool(n, rank):
    """n distinct frames of the config-3 mix (seeded by run/camcol/filter/field), with their blot rects."""
    import lfd_b200
    from lfd_b200.removestars import star_rects
    DEFAULT_REMOVESTARS = lfd_b200.default_params()[2]
    DEFAULT_REMOVESTARS = {k: v for k, v in DEFAULT_REMOVESTARS.items() if k != "debug"}
    frames, cats, rects, kinds = [], [], [], []
    field = 11
    while len(frames) < n:
        flt = synth.FILTERS[len(frames) % 5]
        kind, seed = synth.case_for_frame(2888, 1 + rank % 6, flt, field + 1000 * (rank // 6))
        img, cat = synth.make_case(kind, seed)
        frames.append(img); cats.append(cat); kinds.append(kind)
        rects.append(star_rects(cat, flt, img.shape, **DEFAULT_REMOVESTARS))
        field += 1
    return frames, cats, rects, kinds


class ClockSampler:
    """SM clock + throttle reasons sampled every few ms DURING the timed regions (NVML in a thread; the
    B200_PROFILING.md nvidia-smi query is the fallback).  pause()/resume() bracket untimed sections."""
    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"),
               (0x80, "hw_power_brake_slowdown"))

    def __init__(self, gpu, period_s=0.004):
        import threading
        self.gpu, self.period = gpu, period_s
        self.sm, self.bits, self.smax = [], 0, None
        self._run = threading.Event()
        self._stop = threading.Event()
        self._th = None
        self._nv = None
        self.source = None
        try:
            import pynvml
            pynvml.nvmlInit()
            dev = None
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(gpu).uuid)
                dev = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                dev = pynvml.nvmlDeviceGetHandleByIndex(gpu)
            self._nv, self._dev = pynvml, dev
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(dev, pynvml.NVML_CLOCK_SM))
            self.source = "nvml"
        except Exception:
            self._nv = None

    def _loop(self):
        nv, dev = self._nv, self._dev
        while not self._stop.is_set():
            if self._run.is_set():
                try:
                    self.sm.append(float(nv.nvmlDeviceGetClockInfo(dev, nv.NVML_CLOCK_SM)))
                    self.bits |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(dev))
                except Exception:
                    pass
            time.sleep(self.period)

    def start(self):
        import threading
        if self._nv is not None:
            self._th = threading.Thread(target=self._loop, daemon=True)
            self._th.start()
        else:
            self._smi_start()
        self.resume()

    def resume(self):
        self._run.set()

    def pause(self):
        self._run.clear()

    # nvidia-smi fallback (one process for the whole run; coarse)
    def _smi_start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self._f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self._p = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                        "-lms", "20"], stdout=self._f, stderr=subprocess.DEVNULL)
            self.source = "nvidia-smi"
        except Exception:
            self._p = None

    def stop(self):
        self._stop.set()
        self.pause()
        if self._th is not None:
            self._th.join(timeout=2)
        elif getattr(self, "_p", None):
            self._p.terminate()
            try:
                self._p.wait(timeout=5)
            except Exception:
                self._p.kill()
            self._f.flush(); self._f.seek(0)
            for line in self._f:
                t = [x.strip() for x in line.split(",")]
                try:
                    self.sm.append(float(t[0])); self.smax = float(t[1])
                except (ValueError, IndexError):
                    continue
                for (bit, _), v in zip(self.REASONS[:4], t[2:6]):
                    if v.lower().startswith("active"):
                        self.bits |= bit
            os.unlink(self._f.name)
        out = {"sm_mhz": None, "sm_max_mhz": self.smax, "reasons": [n for b, n in self.REASONS if self.bits & b],
               "samples": len(self.sm), "source": self.source}
        if self.sm:
            out["sm_mhz"] = statistics.median(self.sm)
            out["sm_min_mhz"] = min(self.sm)
        return out


# ----------------------------------------------------------------------------------------------
# CPU reference leg: the oracle's restatement of the reference's call sequence on cv2, all host cores
# ----------------------------------------------------------------------------------------------
_CPU_PARAMS = (None, None)      # (params_bright, params_dim) of the workload, inherited by the forked workers


_CPU_POOL = None                # (frames, cats): inherited by the forked workers, so a job is an index, not 12 MB of pickle


def _cpu_worker(i):
    import cv2
    cv2.setNumThreads(1)
    from oracle import ref_pipeline as rp
    frames, cats = _CPU_POOL
    img, cat, flt = frames[i % len(frames)], cats[i % len(frames)], synth.FILTERS[i % 5]
    t = time.perf_counter()
    try:
        rp.process_frame(img.copy(), cat, flt, _CPU_PARAMS[0], _CPU_PARAMS[1])
    except Exception:   # noqa: BLE001 - a frame the reference would log to errors.txt still costs its time
        pass
    return time.perf_counter() - t


def _cpu_worker_files(args):
    """Figure (ii) of SURVEY.md 8(d): the same frame from FILES - FITS image + header read, photoObj table read and
    remove_stars' catalog loop, then the pipeline (detecttrails.py:113-131)."""
    import cv2
    cv2.setNumThreads(1)
    from lfd_b200 import fitsio_lite
    from oracle import ref_pipeline as rp
    fpath, opath, flt = args
    t = time.perf_counter()
    img = fitsio_lite.read(fpath)
    fitsio_lite.read_header(fpath)
    cat, _h = fitsio_lite.read(opath, header="True")
    try:
        rp.process_frame(np.ascontiguousarray(img, np.float32), cat, flt, _CPU_PARAMS[0], _CPU_PARAMS[1])
    except Exception:   # noqa: BLE001
        pass
    return time.perf_counter() - t


def cpu_frames_per_s_files(frames, cats, nframes, cores):
    """Frames/s of the oracle pipeline fed from FITS files in a temporary directory (page cache), all cores."""
    import multiprocessing as mp
    import shutil
    from lfd_b200 import fitsio_lite
    root = tempfile.mkdtemp(prefix="lfd_b200_cpu_")
    try:
        nd = len(frames)                                  # the same frames, in the same order, as the compute-only leg
        for i in range(nd):
            fitsio_lite.write_image(os.path.join(root, "frame%d.fits" % i), frames[i], dict(synth.DEFAULT_HEADER))
            fitsio_lite.write_bintable(os.path.join(root, "photoObj%d.fits" % i), cats[i])
        jobs = [(os.path.join(root, "frame%d.fits" % (i % nd)), os.path.join(root, "photoObj%d.fits" % (i % nd)), synth.FILTERS[i % 5])
                for i in range(nframes)]
        with mp.get_context("fork").Pool(cores) as pool:
            pool.map(_cpu_worker_files, jobs[:cores])
            t0 = time.perf_counter()
            pool.map(_cpu_worker_files, jobs, chunksize=1)
            dt = time.perf_counter() - t0
        return nframes / dt, dt
    finally:
        shutil.rmtree(root, ignore_errors=True)


def cpu_frames_per_s(frames, cats, nframes, cores, repeat=1):
    """Wall-clock frames/s of the oracle pipeline over `nframes` frames on `cores` processes (frames already decoded in
    RAM and shared with the workers by fork, so no per-job transfer is timed)."""
    global _CPU_POOL
    import multiprocessing as mp
    _CPU_POOL = (frames, cats)
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        pool.map(_cpu_worker, range(cores))          # warm the workers (imports, page-in)
        best = None
        for _ in range(repeat):
            t0 = time.perf_counter()
            pool.map(_cpu_worker, range(nframes), chunksize=1)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
    return nframes / best, best


def run_reference(args):
    global _CPU_PARAMS
    rank = env_int("RANK", 0)
    if rank != 0:
        return 0
    if args.workload == "config5":
        return run_reference_config5(args)
    WORKLOAD, pb_, pd_ = workload_params(args)
    _CPU_PARAMS = (pb_, pd_)
    cores = os.cpu_count() or 1
    frames, cats, _rects, _kinds = make_pool(64, 0)      # the same 64-frame pool rank 0 of our arm uses
    cal_value, _ = cpu_frames_per_s(frames, cats, max(2 * cores, 8), cores)
    per_step = int(min(max(cal_value * 4.0, 2 * cores), 2048))   # ~4 s of all-core CPU work per step
    import multiprocessing as mp
    global _CPU_POOL
    _CPU_POOL = (frames, cats)
    with mp.get_context("fork").Pool(cores) as pool:
        for _ in range(max(args.warmup, 1)):
            pool.map(_cpu_worker, range(cores))
        t0 = time.perf_counter()
        for _ in range(args.steps):
            pool.map(_cpu_worker, range(per_step), chunksize=1)
        dt = time.perf_counter() - t0
    value = per_step * args.steps / dt
    import cv2
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32/u8", "data": "synthetic",
        "config": {"workload": WORKLOAD, "frame": [H, W], "frames_per_step": per_step, "cv2": cv2.__version__, "numpy": np.__version__},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": cores, "kind": "port",
                         "sample": "%d frames/step x %d steps of the %s pool, oracle/ref_pipeline.py (reference call sequence on cv2 %s), "
                                   "multiprocessing.Pool(%d), cv2.setNumThreads(1); the workers inherit the decoded frames by fork, a job "
                                   "is an index (round 1 pickled 12 MB per job inside the timed region, which halved this figure)"
                                   % (per_step, args.steps, WORKLOAD, cv2.__version__, cores)},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


# ----------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------
def bind_to_gpu_numa_node(gpu):
    """Pin this rank's host threads to the CPUs NVML reports as local to its GPU, so that the pinned staging buffers
    are first-touched on the NUMA node the GPU's PCIe root hangs off (matters once several ranks pull 55 GB/s each)."""
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        uuid = str(torch.cuda.get_device_properties(gpu).uuid)
        dev = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(dev, (ncpu + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:   # noqa: BLE001 - best effort
        pass
    return None


def dropin_leg(device, ndistinct=32, nfields=1024, batch=32, verify=True, rank=0, world=1, dist=None):
    """Frames/s of the user-facing call: a synthetic SDSS tree on local disk (FITS frames + photoObj tables),
    lfd_b200.DetectTrails(run=, camcol=, filter=).process() writing results.txt - FITS reads (page cache), catalog
    filtering, pinned staging, H2D, kernels, D2H and the text output all inside the timed region.  `ndistinct`
    synthetic fields are generated and hard-linked up to `nfields` file names per GPU (generation time, not run time).
    Under torchrun every rank calls this: the frame list is sharded over the ranks, rank 0 gathers and writes."""
    import shutil
    import lfd_b200
    nfields *= world                                  # weak scaling: 1024 frames per GPU
    root = os.path.join(tempfile.gettempdir(), "lfd_b200_bench_%d" % env_int("MASTER_PORT", os.getpid() if world == 1 else 0))
    boss = os.path.join(root, "boss")
    photoobj, redux = os.path.join(boss, "photoObj"), os.path.join(boss, "photo", "redux")
    fdir = os.path.join(photoobj, "frames", "301", "2888", "1")
    odir = os.path.join(photoobj, "301", "2888", "1")
    # every rank keeps a share of the host cores for its loader threads
    os.environ["LFD_LOADER_THREADS"] = os.environ.get("LFD_BENCH_LOADERS") or str(max(2, min(12, (os.cpu_count() or 2) // world)))
    try:
        tree = None
        if rank == 0:
            shutil.rmtree(root, ignore_errors=True)
            tree = synth.write_sdss_tree(root, 2888, 1, range(100, 100 + ndistinct), filters=("r",), startfield=100, endfield=100 + nfields)
            for k in range(ndistinct, nfields):
                src = 100 + k % ndistinct
                os.link(os.path.join(fdir, "frame-r-002888-1-%04d.fits" % src), os.path.join(fdir, "frame-r-002888-1-%04d.fits" % (100 + k)))
                os.link(os.path.join(odir, "photoObj-002888-1-%04d.fits" % src), os.path.join(odir, "photoObj-002888-1-%04d.fits" % (100 + k)))
        if dist is not None:
            dist.barrier()
        lfd_b200.setup(boss, photoobj, redux, root)
        best = None
        for rep_i in range(3):                       # first repetition warms the page cache and creates the handles
            out = os.path.join(root, "out%d" % rep_i)
            if rank == 0:
                os.makedirs(out)
            if dist is not None:
                dist.barrier()
            dt = lfd_b200.DetectTrails(run=2888, camcol=1, filter="r", savepath=out, batch=batch, device=device)
            t0 = time.perf_counter()
            dt.process()
            if dist is not None:
                dist.barrier()                       # the slowest rank ends the run
            el = time.perf_counter() - t0
            if rep_i > 0:
                best = el if best is None else min(best, el)
        if rank != 0:
            return None
        # the host-side ceiling of this leg: the same native ingest calls alone (no H2D, no kernels) over 8 batches
        ingest_only = None
        try:
            from lfd_b200 import _lib, sdssfiles
            pr = {k: v for k, v in lfd_b200.default_params()[2].items() if k != "debug"}
            stg = np.empty((batch, H, W), np.uint32)
            fl = [(2888, 1, "r", 100 + k) for k in range(8 * batch)]
            fp = [sdssfiles.filename("frame", run=r_, camcol=c_, field=f_, filter=fl_) for (r_, c_, fl_, f_) in fl]
            cp = [sdssfiles.filename("photoObj", run=r_, camcol=c_, field=f_) for (r_, c_, fl_, f_) in fl]
            nthr = int(os.environ["LFD_LOADER_THREADS"])
            _lib.ingest_batch(stg, fp[:batch], cp[:batch], ["r"] * batch, nthreads=nthr, **pr)
            t0 = time.perf_counter()
            for b0 in range(0, len(fl), batch):
                _lib.ingest_batch(stg, fp[b0:b0 + batch], cp[b0:b0 + batch], ["r"] * batch, nthreads=nthr, **pr)
            ingest_only = len(fl) / (time.perf_counter() - t0)
        except Exception:   # noqa: BLE001
            pass
        got = open(os.path.join(out, "results.txt")).read()
        nlines = got.count("\n")
        verified = None
        if verify:
            # checker: the oracle's lines for the distinct fields, repeated for the hard-linked names
            from oracle import ref_pipeline as rp
            from oracle.verdicts import verdicts
            from lfd_b200 import fitsio_lite
            src_fields = list(range(100, 100 + ndistinct))
            ref = verdicts([tree["frames"][("r", f)][0] for f in src_fields], [tree["frames"][("r", f)][1] for f in src_fields],
                           ["r"] * ndistinct)
            hdrs = [fitsio_lite.read_header(os.path.join(fdir, "frame-r-002888-1-%04d.fits" % f)) for f in src_fields]
            exp = "".join(rp.result_line(2888, 1, "r", 100 + k, hdrs[k % ndistinct], ref[k % ndistinct][2])
                          for k in range(nfields) if ref[k % ndistinct][0] is True)
            verified = nfields if got == exp else 0
        return {"value": nfields / best, "unit": "frames/s", "frames": nfields, "batch": batch, "detections": nlines,
                "verified": verified, "n_gpus": world,
                "ingest_only_frames_per_s": ingest_only,
                "ingest_note": "ingest_only = the native batch reader alone into pageable memory (page cache -> user copy of 12.2 MB per "
                               "frame plus the catalog filter), no H2D copy competing for host memory bandwidth",
                "how": "DetectTrails(run, camcol, filter).process() on a synthetic tree in %s (%d distinct fields hard-linked to %d, "
                       "%d per GPU): one native call per batch reads the raw FITS payloads into pinned staging and filters the photoObj "
                       "catalogs on %s C++ threads (page cache), ring of three handles per GPU, frame list sharded over the ranks, "
                       "results.txt written by rank 0 in sequential order and checked against the oracle's lines; wall clock of the "
                       "slowest rank, best of 2 after a warm-up pass"
                       % (tempfile.gettempdir(), ndistinct, nfields, nfields // world, os.environ["LFD_LOADER_THREADS"])}
    finally:
        if dist is not None:
            dist.barrier()
        if rank == 0:
            shutil.rmtree(root, ignore_errors=True)


def run_ours(args):
    global _CPU_PARAMS
    import torch
    import torch.distributed as dist
    import lfd_b200
    from lfd_b200 import _lib
    if args.workload == "config5":
        return run_ours_config5(args)

    rank, world, local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    distributed = world > 1
    # one rank per GPU; with more GPUs visible than ranks the ranks are spread over the device indices, because GPUs with
    # neighbouring indices share a host bridge and host->device PCIe is the pipeline's scarce link (lfd_b200/sharding.py)
    from lfd_b200.sharding import spread_device
    local = spread_device(local_rank, world, torch.cuda.device_count())
    torch.cuda.set_device(local)
    orig_affinity = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa_node(local)        # before any pinned allocation (first-touch places the staging pages)
    if distributed:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    B = args.batch

    def barrier():
        torch.cuda.synchronize()
        if distributed:
            dist.barrier()
            torch.cuda.synchronize()

    def reduce_max(x):
        if not distributed:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def reduce_sum(x):
        if not distributed:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    frames, cats, rects, kinds = make_pool(B, rank)
    WORKLOAD, pb, pd = workload_params(args)    # config 3: the drop-in's own defaults (detecttrails.py:202-239)
    _CPU_PARAMS = (pb, pd)
    hA = _lib.Handle(H, W, max_batch=B, device=local)
    hB = _lib.Handle(H, W, max_batch=B, device=local)
    # more than two ranks behind one PCIe host bridge: the ranks of a bridge slot take turns with their batch copies
    # (lfd_b200/sharding.py::h2d_gate_path; None on one or two ranks per bridge)
    from lfd_b200.sharding import apply_h2d_gate
    gate = apply_h2d_gate((hA, hB), local, world, torch.cuda.device_count()) if distributed else None
    for h in (hA, hB):
        h.set_params(pb, pd)
        for i, f in enumerate(frames):
            h.host_frames[i] = f                       # pinned host staging, filled once

    # ---- value: batch resident in HBM -------------------------------------------------------
    res = hA.upload(B, rects)                          # H2D once (+ one untimed run)
    n_detect = sum(r.detected for r in res)
    pipelined = not args.serial_steps
    depth = max(2, args.inflight) if pipelined else 1
    hs2 = [hA, hB] + [_lib.Handle(H, W, max_batch=B, device=local) for _ in range(depth - 2)]
    if pipelined:
        for h in hs2[1:]:
            if h is not hB:
                h.set_params(pb, pd)
                for i, f in enumerate(frames):
                    h.host_frames[i] = f
            h.upload(B, rects)                         # every handle of the pipeline holds the same resident batch

    def resident_loop(steps):
        """K steps back to back.  Pipelined (default): `depth` handles take turns with `depth` steps in flight, so the
        memory-bound head of step k+1 (setup + k_prep) overlaps the latency-bound tail of step k, exactly as consecutive
        batches do in the e2e leg and in the drop-in driver.  --serial-steps: one handle, every step collected before the
        next is launched.  Returns (results of the last step, summed k_prep ms, handle of the last step)."""
        prep = 0.0
        res_last = None
        if not pipelined:
            for _ in range(steps):
                hA.run_resident(B); res_last = hA.wait()
                prep += hA.timings()[1][1]
            return res_last, prep, hA
        for k in range(steps):
            if k >= depth:                             # the handle is still busy with step k - depth: collect it first
                hs2[k % depth].wait()
                prep += hs2[k % depth].timings()[1][1]
            hs2[k % depth].run_resident(B)
        for k in range(max(steps - depth, 0), steps):  # drain, oldest first
            res_last = hs2[k % depth].wait()
            prep += hs2[k % depth].timings()[1][1]
        return res_last, prep, hs2[(steps - 1) % depth]

    resident_loop(max(args.warmup, 3))
    sampler = ClockSampler(local)
    stage_ms = None
    barrier()
    sampler.start()
    l0 = sum(h.kernel_launches() for h in hs2)
    t0 = time.perf_counter()
    hA.timer_mark(0)
    last_res, prep_ms_sum, h_last = resident_loop(args.steps)   # k_prep runs before the passes fork: its bracket is clean
    res_resident = [bytes(r) for r in last_res]
    h_last.timer_mark(1)
    dev_ms = hA.timer_elapsed_ms(0, h_last, 1)        # CUDA events on the library's streams, first launch -> last result
    torch.cuda.synchronize()
    if distributed:
        dist.barrier()
    wall_s = time.perf_counter() - t0
    sampler.pause()
    launches = sum(h.kernel_launches() for h in hs2) - l0
    for h in hs2[2:]:
        h.close()
    elapsed = reduce_max(dev_ms) / 1e3
    wall_s = reduce_max(wall_s)
    counters = hA.counters()
    value = world * B * args.steps / elapsed
    # kernel brackets: the SAME K steps again with a CUDA event on each side of the launches that carry the step (inside
    # the captured graph, all four streams running).  The ~50 extra event nodes cost ~5 % of the step, which is why the
    # headline region above runs without them; `bracketed_ms_per_step` says what this second region took.
    kacc = {}                                         # (kernel, pass) -> [ms summed over launches and steps, launches]
    for _ in range(2):
        hA.run_resident(B, flags=_lib.KERNEL_TIMES); hA.wait()
    hA.timer_mark(0)
    for _ in range(args.steps):
        hA.run_resident(B, flags=_lib.KERNEL_TIMES); hA.wait()
        for name, p_, ms, nl in hA.kernel_times():
            a = kacc.setdefault((name, p_), [0.0, 0])
            a[0] += ms; a[1] += nl
    hA.timer_mark(1)
    bracketed_ms_per_step = hA.timer_elapsed_ms(0, hA, 1) / args.steps
    # per-stage table: a few extra steps with the two passes serialised on one stream (in the timed loop above
    # the bright and the dim pass overlap on two streams, so per-stage brackets would overlap too)
    n_serial = 5
    for _ in range(n_serial):
        hA.run_resident(B, flags=_lib.SERIAL_PASSES); hA.wait()
        tm = hA.timings()
        stage_ms = tm if stage_ms is None else [(n, a + b) for (n, a), (_, b) in zip(stage_ms, tm)]
    serial_ms = sum(ms for _, ms in stage_ms) / n_serial

    if args.profile:
        if rank == 0:
            print(json.dumps({"metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
                              "warmup": args.warmup, "ms_per_step": 1e3 * elapsed / args.steps, "profile_only": True,
                              "config": {"workload": WORKLOAD, "frames_per_step_per_gpu": B},
                              "stages": [{"stage": n, "ms_per_step": ms / n_serial} for n, ms in stage_ms]}))
            if args.dump_outputs:
                dump_arrays(args.dump_outputs, result_arrays("resident", res_resident))
        sampler.stop()
        return 0

    # ---- e2e: host frames -> device -> results, double-buffered over two handles -------------
    def e2e_loop(steps):
        hs = (hA, hB)
        hs[0].submit(B, rects)
        for k in range(1, steps):
            hs[k & 1].submit(B, rects)
            hs[(k - 1) & 1].wait()
        return hs[(steps - 1) & 1].wait()
    e2e_loop(max(args.warmup, 2))
    barrier()
    l1 = hA.kernel_launches() + hB.kernel_launches()
    sampler.resume()
    t0 = time.perf_counter()
    hA.timer_mark(2)
    res_e2e = [bytes(r) for r in e2e_loop(args.steps)]
    last = (hA, hB)[(args.steps - 1) & 1]
    last.timer_mark(3)
    e2e_dev_ms = hA.timer_elapsed_ms(2, last, 3)      # device clock: first H2D enqueued -> last result copied back
    torch.cuda.synchronize()
    if distributed:
        dist.barrier()
    e2e_wall = reduce_max(time.perf_counter() - t0)
    clocks = sampler.stop()
    e2e_elapsed = reduce_max(e2e_dev_ms) / 1e3
    launches_e2e = hA.kernel_launches() + hB.kernel_launches() - l1
    e2e_value = world * B * args.steps / e2e_elapsed
    # H2D-only time (PCIe) reported separately
    t0 = time.perf_counter()
    for _ in range(3):
        hA._ck(hA._L.lfd_upload(hA.h, None, B, None, None, 0))
    torch.cuda.synchronize()
    import ctypes
    h2d_s = (time.perf_counter() - t0) / 3
    rect_bytes = int(sum(len(r) for r in rects) * 16 + (B + 1) * 4)
    h2d_bytes = B * N * 4 + rect_bytes
    d2h_bytes = B * (ctypes.sizeof(_lib.Result) + 96) + 128

    launches_total = int(reduce_sum(launches + launches_e2e))
    os.sched_setaffinity(0, orig_affinity)     # the CPU baseline and the drop-in leg use every host core
    if args.dump_outputs and rank == 0:
        dump_arrays(args.dump_outputs, {**result_arrays("resident", res_resident), **result_arrays("e2e", res_e2e)})

    # ---- verify: the results of the LAST TIMED step of both legs against the oracle, outside the timed regions ----
    verified = mismatches = None
    if not args.no_verify:
        from oracle.verdicts import device_verdict, verdicts
        filters = [synth.FILTERS[i % 5] for i in range(B)]
        ref = verdicts(frames, cats, filters, pb, pd, None, cores=max((os.cpu_count() or 1) // world, 1))
        ok = 0
        for i in range(B):
            want = tuple(ref[i])
            got_r = device_verdict(_lib.Result.from_buffer_copy(res_resident[i]), (H, W))
            got_e = device_verdict(_lib.Result.from_buffer_copy(res_e2e[i]), (H, W))
            if got_r == want and got_e == want:
                ok += 1
            else:
                print("verify: rank %d frame %d (%s): resident %s, e2e %s, oracle %s" % (rank, i, kinds[i], got_r, got_e, want), file=sys.stderr)
        verified = int(reduce_sum(ok))
        mismatches = int(reduce_sum(B - ok))

    # ---- the drop-in itself: FITS files on disk -> DetectTrails(...).process() -> results.txt; under torchrun the frame
    # list is sharded over the ranks (lfd_b200/sharding.py) and rank 0 writes the file, so every rank takes part ----
    try:
        smem_peak = hA.smem_atomic_peak()            # micro-kernel: conflict-free shared-memory atomics on all SMs
    except Exception:   # noqa: BLE001
        smem_peak = None
    dropin = None
    if not args.no_dropin and args.workload == "config3":
        hA.close(); hB.close()                       # the legs above are done: free their 30 GB before the ring is built
        try:
            dropin = dropin_leg(local, verify=not args.no_verify, rank=rank, world=world, dist=dist if distributed else None)
        except Exception as e:   # noqa: BLE001 - an extra, never fatal for the contract line
            dropin = {"error": "%s: %s" % (type(e).__name__, e)}
            if distributed:
                raise

    if rank != 0:
        if distributed:
            dist.destroy_process_group()
        return 0

    # ---- roofline: the TIME-DOMINANT kernel of the timed region + the table of all bracketed kernels ----------------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak = json.load(open(peaks_path))["hbm_gbs"]; peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak = 6650.0; peak_src = "fallback (B200_PROFILING.md)"
    stage_ms = [(n, ms / n_serial) for n, ms in stage_ms]
    per = dict(stage_ms)
    n_bright, n_dim = counters["frames_bright_run"], counters["frames_dim_run"]
    has_erode = pd.get("erodeKernel") is not None
    # ALGORITHMIC bytes per frame (SURVEY.md 8(d): one compulsory read of the stage input + one write of its output):
    #   S1 prep 4N read + 1N write per pass (one launch produces both passes: 4N + 2N), S2 LUT apply 2N, S3 erode 2N
    #   (dim), S4 dilate 2N, S5 Sobel+NMS 2N, S6 labelling 9N (below).  Rectangles / Hough work on run lists and
    #   shared-memory accumulators: they carry measured DRAM bytes only.  A pass is charged the frames it ran on.
    alg_frame = {("k_prep", 0): 6 * N, ("k_morph_march", 0): 4 * N, ("k_morph_march", 1): (6 if has_erode else 4) * N,
                 ("k_nms_march", 0): 2 * N, ("k_nms_march", 1): 2 * N}
    # what THIS design has to move per frame for the same stages (the LUT is applied inside the morphology kernel, erode and
    # dilate share one pass over the plane, NMS writes two 1-bit masks): the honest denominator for "how far from HBM"
    design_frame = {("k_prep", 0): 6 * N, ("k_morph_march", 0): 2 * N + N // 8, ("k_morph_march", 1): 2 * N + N // 8,
                    ("k_nms_march", 0): N + N // 4, ("k_nms_march", 1): N + N // 4}
    # measured DRAM traffic (dram__bytes_read.sum + dram__bytes_write.sum per 64-frame step) of the newest committed ncu list
    import glob
    measured = {}
    measured_src = None
    for tr_path in sorted(glob.glob(os.path.join(ROOT, "profiles", "traffic_r*.json")), reverse=True):
        try:
            t = json.load(open(tr_path))
            if "per_step_bytes" in t and t.get("batch") == B and t.get("workload", "config3") == args.workload:
                measured, measured_src = t["per_step_bytes"], "profiles/" + os.path.basename(tr_path)
                break
        except Exception:
            pass
    runs_per_frame_pass = {"fg": counters["runs_fg"] / max(n_bright + n_dim, 1), "bg": counters["runs_bg"] / max(n_bright + n_dim, 1)}
    for p_ in (0, 1):
        # S6 (labelling, fg + bg): read 1N, write two int32 label planes = 9N per pass in the survey's model; this design
        # labels RUNS: the band kernel reads the 1-bit mask (N/8) and the per-word run prefix (N/16) and writes ~12 B per run
        alg_frame[("k_ccl_band(fg)", p_)] = 5 * N
        alg_frame[("k_ccl_band(bg)", p_)] = 4 * N
        for kind in ("fg", "bg"):
            design_frame[("k_ccl_band(%s)" % kind, p_)] = N // 8 + N // 16 + int(12 * runs_per_frame_pass[kind])
    frames_of_pass = {0: n_bright, 1: n_dim}
    ktable = [{"kernel": "k_prep", "pass": "both", "ms_per_step": prep_ms_sum / args.steps, "launches_per_step": 1,
               "alg_bytes_per_step": B * alg_frame[("k_prep", 0)], "design_bytes_per_step": B * design_frame[("k_prep", 0)]}]
    for (name, p_), (ms, nl) in sorted(kacc.items()):
        e = {"kernel": name, "pass": ("bright", "dim")[p_], "ms_per_step": ms / args.steps, "launches_per_step": nl / args.steps}
        if (name, p_) in alg_frame:
            e["alg_bytes_per_step"] = frames_of_pass[p_] * alg_frame[(name, p_)]
            e["design_bytes_per_step"] = frames_of_pass[p_] * design_frame[(name, p_)]
        ktable.append(e)
    roofline, ktable = build_roofline(ktable, peak, peak_src, measured, measured_src, stage_ms, n_serial, bracketed_ms_per_step)
    stage_report = []
    alg_stage = {"lut+morph": 4 * N, "dim:lut+morph": (6 if has_erode else 4) * N, "sobel+nms": 2 * N}
    for name, ms in stage_ms:
        entry = {"stage": name, "ms_per_step": round(ms, 4)}
        key = name.split(":")[-1].split("(")[0]
        full = name.split("(")[0]
        nfr = n_bright if name.startswith("bright") else n_dim if name.startswith("dim") else B
        if name.startswith("prep"):
            entry.update(alg_bytes=B * 6 * N)
        elif full in alg_stage or key in alg_stage:
            entry.update(alg_bytes=nfr * alg_stage.get(full, alg_stage.get(key)))
        if entry.get("alg_bytes") and ms > 0:
            entry["gbs"] = entry["alg_bytes"] / (ms * 1e6)
            entry["frac_of_hbm_peak"] = entry["gbs"] / peak
        stage_report.append(entry)
    hough_ms = per["bright:hough"] + per["dim:hough"]
    vote_ms = sum(e["ms_per_step"] for e in ktable if e["kernel"] == "k_hough_vote")

    # ---- CPU baseline on this box's host cores (bounded sample) -------------------------------
    cores = os.cpu_count() or 1
    cpu_baseline = None
    if world == 1:
        # bounded sample: calibrate on 2 frames per core, then size the timed sample for ~12 s of wall clock
        cal_value, _ = cpu_frames_per_s(frames, cats, max(2 * cores, 8), cores)
        sample = int(min(max(cal_value * 12.0, 4 * cores), 4096))
        cpu_value, cpu_s = cpu_frames_per_s(frames, cats, sample, cores)
        import cv2
        # figure (ii) of SURVEY.md 8(d): the same pipeline fed from files (FITS image + header + photoObj table reads and
        # remove_stars' catalog loop inside the timed region), ~6 s of wall clock
        io_sample = int(min(max(cal_value * 6.0, 2 * cores), 2048))
        io_value, io_s = cpu_frames_per_s_files(frames, cats, io_sample, cores)
        cpu_baseline = {"value": cpu_value, "unit": "frames/s", "cores": cores, "kind": "port",
                        "sample": "%d frames of the same pool, oracle/ref_pipeline.py (reference call sequence on cv2 %s), "
                                  "multiprocessing.Pool(%d), cv2.setNumThreads(1), %.1f s; the unmodified reference cannot travel to the "
                                  "GPU box (pure Python under /root/reference), the port calls the same cv2 binary at the same call sites"
                                  % (sample, cv2.__version__, cores, cpu_s),
                        "value_with_file_io": io_value,
                        "sample_with_file_io": "%d frames read from FITS files in %s (image + header + photoObj table, page cache) and run "
                                               "through remove_stars + both passes, %.1f s" % (io_sample, tempfile.gettempdir(), io_s)}

    line = {
        "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * elapsed / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32/u8", "data": "synthetic",
        "config": {"workload": WORKLOAD, "frame": [H, W], "frames_per_step_per_gpu": B, "pool": "B distinct frames per rank "
                   "(sparse/dense/trail/satellite mix, seeded), inputs %.0f MB per step > L2 (126 MB), no L2 flush" % (B * N * 4 / 1e6),
                   "kinds": {k: kinds.count(k) for k in sorted(set(kinds))}, "detections_per_batch": int(n_detect),
                   "parallelism": "frame-sharded x%d, no collective" % world, "host_cpus_bound_per_rank": numa,
                   "cuda_device_of_rank0": local, "device_map": os.environ.get("LFD_DEVICE_MAP", "spread"),
                   "h2d_gate_of_rank0": gate},
        "timing": ("resident leg: K steps issued back to back on %d handles holding the same resident batch, %d steps in flight " % (depth, depth) +
                   "(the head of step k+1 overlaps the tail of step k; --serial-steps measures one step at a time); " if pipelined else
                   "resident leg: one handle, every step collected before the next is launched; ") +
                  "CUDA events on the library's stream around the K steps (max over ranks); wall clock alongside: "
                  "%.3f ms/step resident, %.3f ms/step e2e" % (1e3 * wall_s / args.steps, 1e3 * e2e_wall / args.steps),
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                "ms_per_step": 1e3 * e2e_elapsed / args.steps, "h2d_only_ms_per_step": 1e3 * h2d_s,
                "h2d_gbs": h2d_bytes / h2d_s / 1e9, "how": "lfd_submit from pinned host staging + lfd_wait, two handles double-buffered"},
        "gpu_launches": launches_total,
        "verified": verified, "verify_mismatches": mismatches,
        "verify_note": "verdict (detected, pass, end points) of every frame of the last timed step of the resident leg and of the "
                       "e2e leg == oracle/ref_pipeline.py::process_frame on the same frame (all ranks; checker only, untimed)",
        "roofline": roofline,
        "kernels": ktable,
        "measured_dram": {"source": measured_src, "per_step_bytes_both_passes": measured or None,
                          "note": "dram__bytes_read.sum + dram__bytes_write.sum per 64-frame step from the committed ncu list; "
                                  "the design's own byte count is 12N per frame (prep 6N, morph 2 x 2N, NMS 2 x 1N + masks)"},
        "stages": stage_report,
        "stages_note": "per-stage CUDA-event times of %d extra steps with the passes serialised (LFD_SERIAL_PASSES), %.3f ms/step; "
                       "in the timed region the bright and dim passes overlap on two streams" % (n_serial, serial_ms),
        "hough": {"ms_per_step": hough_ms, "vote_kernel_ms_per_step_live": vote_ms, "votes_per_step": counters["votes"],
                  "gvotes_per_s": counters["votes"] / (hough_ms * 1e6) if hough_ms > 0 else None,
                  "smem_atomics_issued_per_step": counters.get("hough_smem_atomics"),
                  "votes_per_atomic": (counters["votes"] / counters["hough_smem_atomics"]) if counters.get("hough_smem_atomics") else None,
                  "gatomics_per_s": (counters["hough_smem_atomics"] / (vote_ms * 1e6)) if counters.get("hough_smem_atomics") and vote_ms > 0 else None,
                  "frames_hough": counters["frames_hough"],
                  "smem_atomic_peak_gops": smem_peak,
                  "rho": [float(pb["houghMethod"]), float(pd["houghMethod"])],
                  "note": "votes = non-zero pixels x 180 angles of the frames that reach HoughLines. The kernel issues one shared-memory "
                          "atomic per (32-pixel mask word, angle, rho bin), not one per vote, so its binding resource is not the atomic "
                          "unit (gatomics_per_s against smem_atomic_peak_gops) but instruction issue: cvRound(x cos + y sin) per "
                          "(word, angle), FP32 magic-number conversions since round 2 instead of the XU pipe (profiles/r02_sass_summary.md)"},
        "counters": counters,
        "cpu_baseline": cpu_baseline,
        "dropin_e2e": dropin,
    }
    print(json.dumps(line))
    if distributed:
        dist.destroy_process_group()
    return 0


# ----------------------------------------------------------------------------------------------
# config 5: Hough / Canny stage microbenchmark on 4096 x 4096 (BASELINE.json configs[4], SURVEY.md 8(d))
# ----------------------------------------------------------------------------------------------
C5_SIZE = 4096
C5_DENSITIES = (0.001, 0.003, 0.01, 0.03, 0.10)
C5_RHOS = (20.0, 5.0, 1.0)
C5_THETAS = (np.pi / 180, np.pi / 360, np.pi / 720, np.pi / 1440)


def c5_image(density, seed):
    """uint8 4096 x 4096: Bernoulli non-zero pixels at `density` plus three straight lines (values 1..255)."""
    rng = np.random.default_rng(seed)
    img = (rng.random((C5_SIZE, C5_SIZE)) < density).astype(np.uint8) * rng.integers(1, 256, (C5_SIZE, C5_SIZE), dtype=np.uint8)
    for k in range(3):
        x0, y0, x1, y1 = rng.integers(0, C5_SIZE, 4)
        n = int(max(abs(int(x1) - int(x0)), abs(int(y1) - int(y0)))) + 1
        xs = np.rint(np.linspace(x0, x1, n)).astype(np.int64); ys = np.rint(np.linspace(y0, y1, n)).astype(np.int64)
        img[ys, xs] = 255
    return img


def c5_cases(quick=False):
    """(density, rho, theta) grid: the full density x rho sweep at theta = pi/180 plus the theta sweep at 1 % density."""
    cases = [(dn, rho, C5_THETAS[0]) for dn in C5_DENSITIES for rho in C5_RHOS]
    cases += [(0.01, rho, th) for th in C5_THETAS[1:] for rho in (20.0, 1.0)]
    return cases[:4] if quick else cases


def _c5_cpu(args):
    import cv2
    cv2.setNumThreads(1)
    dn, rho, th, seed = args
    img = c5_image(dn, seed)
    t = time.perf_counter()
    lines = cv2.HoughLines(img, rho, th, 1)
    dt = time.perf_counter() - t
    t = time.perf_counter()
    cv2.Canny(img, 0, 255)
    dc = time.perf_counter() - t
    return int(np.count_nonzero(img)), 0 if lines is None else len(lines), dt, dc


def run_reference_config5(args):
    """cv2.HoughLines / cv2.Canny on the same images, one case per host core at a time (votes/s over the wall clock)."""
    import multiprocessing as mp
    import cv2
    cores = os.cpu_count() or 1
    cases = c5_cases()
    jobs = [(dn, rho, th, 100 + i) for i, (dn, rho, th) in enumerate(cases)]
    with mp.get_context("fork").Pool(min(cores, len(jobs))) as pool:
        t0 = time.perf_counter()
        out = pool.map(_c5_cpu, jobs, chunksize=1)
        wall = time.perf_counter() - t0
    votes = 0.0
    per_case = []
    for (dn, rho, th), (nnz, nl, dt, dc) in zip(cases, out):
        na = int(np.floor(np.pi / th)) + 1
        if abs(np.pi - (na - 1) * th) < th / 2:
            na -= 1
        votes += nnz * na
        per_case.append({"density": dn, "rho": rho, "theta_div": int(round(np.pi / th)), "nnz": nnz, "lines": nl,
                         "hough_ms": 1e3 * dt, "gvotes_per_s_1core": nnz * na / dt / 1e9, "canny_ms": 1e3 * dc})
    value = votes / sum(c["hough_ms"] for c in per_case) * 1e3 / 1e9 * min(cores, len(jobs))
    line = {"impl": "reference", "metric": "Hough Gvotes/s (4096x4096 microbench, cv2.HoughLines)", "value": value, "unit": "Gvotes/s",
            "n_gpus": args.gpus, "steps": 1, "warmup": 0, "ms_per_step": 1e3 * wall, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32/int32", "data": "synthetic",
            "config": {"workload": WORKLOADS["config5"], "image": [C5_SIZE, C5_SIZE], "cases": len(cases), "cv2": cv2.__version__},
            "cpu_baseline": {"value": value, "unit": "Gvotes/s", "cores": min(cores, len(jobs)), "kind": "reference",
                             "sample": "cv2.HoughLines on the %d microbench images, one case per core (votes of all cases / summed "
                                       "single-core Hough time x cores)" % len(cases)},
            "e2e": {"value": value, "unit": "Gvotes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "cases": per_case}
    print(json.dumps(line))
    return 0


def run_ours_config5(args):
    """lfd_hough_lines / lfd_canny on 4096 x 4096 images (device times of the kernels from CUDA events on the library's
    stream; the image upload and the line download are outside them), every case checked against cv2 (lines bit for bit)."""
    import torch
    from lfd_b200 import _lib
    local = env_int("LOCAL_RANK", 0)
    if env_int("RANK", 0) != 0:
        return 0
    torch.cuda.set_device(local)
    h = _lib.Handle(C5_SIZE, C5_SIZE, max_batch=1, device=local, max_runs=1 << 23, max_components=1 << 20)
    import lfd_b200
    pb, pd, _ = lfd_b200.default_params()
    h.set_params(pb, pd)
    sampler = ClockSampler(local)
    sampler.start()
    cases = c5_cases(quick=args.quick)
    reps = args.steps
    rows, verified, launches0 = [], 0, h.kernel_launches()
    tot_votes = tot_ms = 0.0
    try:
        import cv2
        cv2.setNumThreads(max(os.cpu_count() or 1, 1))
    except Exception:   # noqa: BLE001
        cv2 = None
    for i, (dn, rho, th) in enumerate(cases):
        img = c5_image(dn, 100 + i)
        for _ in range(max(args.warmup, 3) if i == 0 else 1):
            h.hough_lines(img, rho, th, 1, max_lines=0)
        best = None
        for _ in range(reps):
            h.hough_lines(img, rho, th, 1, max_lines=0)          # votes + peaks; the full sort only runs for the check below
            tm = [ms for _n, ms in h.timings()[:4]]
            if best is None or tm[1] < best[1]:
                best = tm
        cnt = h.counters()
        nlines = h.last_n_lines
        row = {"density": dn, "rho": rho, "theta_div": int(round(np.pi / th)), "nnz": cnt["nnz_equ"], "votes": cnt["votes"],
               "lines": nlines, "compact_ms": best[0], "vote_ms": best[1], "peaks_ms": best[2],
               "gvotes_per_s": cnt["votes"] / (best[1] * 1e6), "smem_atomics": cnt["hough_smem_atomics"],
               "votes_per_atomic": cnt["votes"] / max(cnt["hough_smem_atomics"], 1),
               "gatomics_per_s": cnt["hough_smem_atomics"] / (best[1] * 1e6)}
        if not args.no_verify and cv2 is not None:
            ref = cv2.HoughLines(img, rho, th, 1)
            if nlines <= 400000:                                 # full line list, bit for bit (single-CTA sort: kept to small lists)
                lines, _ = h.hough_lines(img, rho, th, 1)
                ok = (ref is None and lines is None) or (ref is not None and lines is not None and np.array_equal(ref, lines))
                row["check"] = "lines"
            else:                                                # huge peak lists of the noise images: the count must agree
                ok = ref is not None and len(ref) == nlines
                row["check"] = "count"
            row["matches_cv2"] = bool(ok)
            verified += int(ok)
        # Canny on the same image (Sobel + NMS kernel, hysteresis by run CCL)
        if th == C5_THETAS[0] and rho == C5_RHOS[0]:
            for _ in range(2):
                edges = h.canny(img, 0, 255)
            tc = [ms for _n, ms in h.timings()[:2]]
            row.update(canny_nms_ms=tc[0], canny_hysteresis_ms=tc[1], canny_gpx_per_s=C5_SIZE * C5_SIZE / ((tc[0] + tc[1]) * 1e6))
            if not args.no_verify and cv2 is not None:
                row["canny_matches_cv2"] = bool(np.array_equal(edges, cv2.Canny(img, 0, 255)))
        rows.append(row)
        tot_votes += cnt["votes"]; tot_ms += best[1]
    clocks = sampler.stop()
    try:
        smem_peak = h.smem_atomic_peak()
    except Exception:   # noqa: BLE001
        smem_peak = None
    base = [r for r in rows if r["rho"] == 20.0 and r["theta_div"] == 180]
    fine = [r for r in rows if r["rho"] == 1.0 and r["theta_div"] == 180]
    line = {"metric": "Hough Gvotes/s (4096x4096 microbench, vote kernel)", "value": tot_votes / (tot_ms * 1e6), "unit": "Gvotes/s",
            "n_gpus": 1, "steps": reps, "warmup": max(args.warmup, 3), "ms_per_step": tot_ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32/int32", "data": "synthetic",
            "config": {"workload": WORKLOADS["config5"], "image": [C5_SIZE, C5_SIZE], "cases": len(cases),
                       "densities": list(C5_DENSITIES), "rhos": list(C5_RHOS), "theta_divisors": [int(round(np.pi / t)) for t in C5_THETAS],
                       "timing": "CUDA events on the library's stream around each phase, best of %d repetitions per case; "
                                 "one image = 16.8 MB in, accumulator up to 148 MB (rho 1, theta pi/1440): larger than L2 only for the fine grids" % reps},
            "clocks": clocks, "gpu_launches": h.kernel_launches() - launches0,
            "verified": verified if not args.no_verify else None, "cases_total": len(cases),
            "roofline": {"bound": "hbm", "kernel": "k_hough_vote", "achieved": None, "peak": None, "unit": "GB/s", "frac": None, "traffic": None,
                         "note": "the vote kernel is bound by instruction issue / shared-memory atomics, not by HBM; see gvotes_per_s, gatomics_per_s "
                                 "against smem_atomic_peak_gops and the ncu summaries in profiles/ (r02n_hough_c4_*)"},
            "smem_atomic_peak_gops": smem_peak,
            "gvotes_per_s_rho20_mean": float(np.mean([r["gvotes_per_s"] for r in base])) if base else None,
            "gvotes_per_s_rho1_mean": float(np.mean([r["gvotes_per_s"] for r in fine])) if fine else None,
            "cases": rows}
    print(json.dumps(line))
    if args.dump_outputs:     # per case, what the last timed lfd_hough_lines call counted
        dump_arrays(args.dump_outputs, {"config5_" + k: [r[k] for r in rows] for k in ("nnz", "votes", "lines")})
    h.close()
    return 0


HBM_STAGE_KERNELS = ("k_prep", "k_morph_march", "k_nms_march")
_STAGE_OF = {"k_nms_march": "sobel+nms", "k_morph_march": "lut+morph"}


def _base(kernel):
    return kernel.split("(")[0]


def build_roofline(ktable, peak, peak_src, measured, measured_src, stage_ms, n_serial, bracketed_ms_per_step):
    """The `roofline` object of the JSON line from the table of bracketed kernels (one row per kernel function, pass and
    labelling kind: kernel, pass, ms_per_step, launches_per_step and, where SURVEY.md 8(d) has a byte figure,
    alg_bytes_per_step / design_bytes_per_step).

    The kernel named is the one that carries the most bracketed time of the step, all its launches together (both passes,
    all batch parts, fg and bg labelling) - whichever stage it belongs to; `hbm_stage` repeats the same figures for the
    time-dominant kernel of the streaming stages (prep / morphology / Sobel+NMS), which is where HBM could bind."""
    measured = measured or {}
    for e in ktable:
        e["avg_launch_ms"] = e["ms_per_step"] / max(e["launches_per_step"], 1)
        if "alg_bytes_per_step" in e and e["ms_per_step"] > 0:
            e["gbs"] = e["alg_bytes_per_step"] / (e["ms_per_step"] * 1e6)
            e["frac_of_hbm_peak"] = e["gbs"] / peak
            e["frac_of_hbm_peak_design_bytes"] = e["design_bytes_per_step"] / (e["ms_per_step"] * 1e6) / peak
        if _base(e["kernel"]) in measured:
            e["dram_bytes_per_step_measured_both_passes"] = measured[_base(e["kernel"])]
    ktable = sorted(ktable, key=lambda e: -e["ms_per_step"])
    tot = {}
    for e in ktable:
        tot[_base(e["kernel"])] = tot.get(_base(e["kernel"]), 0.0) + e["ms_per_step"]

    def describe(dom):
        rows = [e for e in ktable if _base(e["kernel"]) == dom]
        ms = sum(e["ms_per_step"] for e in rows)
        nl = sum(e["launches_per_step"] for e in rows)
        out = {"kernel": dom, "ms_per_step": ms, "launches_per_step": nl, "avg_launch_ms": ms / max(nl, 1),
               "traffic": (measured[dom] / nl) if dom in measured and nl else None}
        if all("alg_bytes_per_step" in e for e in rows) and ms > 0:
            ab = sum(e["alg_bytes_per_step"] for e in rows)
            db = sum(e["design_bytes_per_step"] for e in rows)
            out.update(survey_bytes_per_launch=ab / nl, design_bytes_per_launch=db / nl,
                       frac_survey_bytes=ab / (ms * 1e6) / peak, frac_design_bytes=db / (ms * 1e6) / peak)
            if dom in _STAGE_OF:      # the same kernel with nothing else on the GPU: stage brackets of the serialised steps
                ms_alone = sum(m for n_, m in stage_ms if n_.split(":")[-1].startswith(_STAGE_OF[dom]))
                if ms_alone > 0:
                    out["alone"] = {"ms_per_step": ms_alone, "gbs": ab / (ms_alone * 1e6), "frac": ab / (ms_alone * 1e6) / peak,
                                    "frac_design_bytes": db / (ms_alone * 1e6) / peak,
                                    "how": "CUDA-event stage brackets of the %d steps run with LFD_SERIAL_PASSES (one stream, one launch per pass)" % n_serial}
        elif dom in measured and ms > 0:      # no byte figure in SURVEY.md 8(d) for this kernel: the DRAM bytes ncu measured
            out.update(design_bytes_per_launch=measured[dom] / nl, frac_design_bytes=measured[dom] / (ms * 1e6) / peak,
                       bytes_model="measured DRAM bytes of the committed ncu list (SURVEY.md 8(d) has no byte figure for this kernel)")
        return out

    dom = describe(max(tot, key=lambda k: tot[k]))
    hbm = describe(max((k for k in tot if k in HBM_STAGE_KERNELS), key=lambda k: tot[k]))
    # `frac`: SURVEY.md 8(d)'s algorithmic bytes where the stage streams planes the way the survey counts them (prep,
    # morphology, Sobel+NMS); for the run-based labelling (and kernels the survey gives no bytes for) the survey's int32 label
    # planes are never materialised, so the bytes this design has to move are the algorithmic bytes of the kernel
    use_survey = dom["kernel"] in HBM_STAGE_KERNELS and "frac_survey_bytes" in dom
    frac = dom.get("frac_survey_bytes") if use_survey else dom.get("frac_design_bytes")
    per_launch = dom.get("survey_bytes_per_launch") if use_survey else dom.get("design_bytes_per_launch")
    roofline = {"bound": "hbm", "kernel": dom["kernel"],
                "achieved": (per_launch / (dom["avg_launch_ms"] * 1e6)) if per_launch else None, "peak": peak, "unit": "GB/s",
                "frac": frac, "frac_design_bytes": dom.get("frac_design_bytes"), "frac_survey_bytes": dom.get("frac_survey_bytes"),
                "algorithmic_bytes_per_launch": per_launch, "bytes_model": dom.get("bytes_model", "SURVEY.md 8(d)" if use_survey else "design bytes (see note)"),
                "design_bytes_per_launch": dom.get("design_bytes_per_launch"), "survey_bytes_per_launch": dom.get("survey_bytes_per_launch"),
                "traffic": dom["traffic"], "traffic_source": measured_src, "peak_source": peak_src,
                "avg_launch_ms": dom["avg_launch_ms"], "launches_per_step": dom["launches_per_step"], "ms_per_step": dom["ms_per_step"],
                "bracketed_ms_per_step": bracketed_ms_per_step, "alone": dom.get("alone"),
                "hbm_stage": hbm,
                "all_kernel_ms_per_step": {k: round(v, 4) for k, v in sorted(tot.items(), key=lambda kv: -kv[1])},
                "note": "`kernel` is the kernel function with the most bracketed time per step, all its launches together (both "
                        "passes, all batch parts, fg and bg labelling); `hbm_stage` is the time-dominant kernel of the streaming "
                        "stages (prep / morphology / Sobel+NMS) with the same figures. frac_survey_bytes uses SURVEY.md 8(d)'s "
                        "algorithmic bytes (every stage charged one read of its input and one write of its output: LUT apply, erode "
                        "and dilate are three stages there and one pass over the plane here; labelling is charged two int32 label "
                        "planes that a run-based labelling never writes), frac_design_bytes the bytes this design has to move; "
                        "`frac` is the survey figure for the streaming kernels and the design figure otherwise. Durations are CUDA "
                        "events recorded on the launching stream around every launch inside the captured graph, over a second run "
                        "of the same K steps (bracketed_ms_per_step; the event nodes cost a few % so the headline region runs "
                        "without them), with the other three streams running - a launch timed alone is shorter "
                        "(profiles/*ktiming*, profiles/*launch_shares*). No kernel behind k_prep is HBM-bound: the step is "
                        "instruction-issue / latency bound (profiles/inst_*_summary.txt, DESIGN.md 3). `kernels` lists every bracketed kernel."}
    return roofline, ktable


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="config3", choices=sorted(WORKLOADS),
                    help="BASELINE.json config: 3 = camcol mix at the default params (the headline), 4 = high-sensitivity dim "
                         "(15x15 dilation, fine rho), 5 = Hough/Canny microbench on 4096x4096")
    ap.add_argument("--hough-method", type=float, default=1.0, help="config4: params_dim['houghMethod'] (rho resolution, px)")
    ap.add_argument("--quick", action="store_true", help="config5: first four cases only")
    ap.add_argument("--inflight", type=int, default=2, help="resident leg: steps (= handles) in flight (default 2)")
    ap.add_argument("--serial-steps", action="store_true",
                    help="resident leg: collect every step before launching the next (default: two handles, two steps in flight)")
    ap.add_argument("--profile", action="store_true", help="device-resident leg only (target command for ncu)")
    ap.add_argument("--no-dropin", action="store_true", help="skip the DetectTrails-on-FITS-files leg")
    ap.add_argument("--no-verify", action="store_true", help="skip the oracle check of the timed steps' results")
    ap.add_argument("--verify", action="store_true", help="(default) check the timed steps' results against the oracle")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the results of the last timed step as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the results of this project's timed path (--impl ours)")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    # stdout carries exactly ONE line, the JSON: libraries that print to fd 1 while we run (NCCL's version banner,
    # for one) are sent to stderr, and the real stdout is put back for the final print
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    lines = []
    import builtins
    orig_print = builtins.print

    def capture(*a, **k):
        if k.get("file") in (None, sys.stdout):
            lines.append(" ".join(str(x) for x in a))
        else:
            orig_print(*a, **k)
    builtins.print = capture
    try:
        rc = run_reference(args) if args.impl == "reference" else run_ours(args)
    finally:
        builtins.print = orig_print
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        os.close(real_stdout)
    for ln in lines:
        print(ln)
    sys.stdout.flush()
    return rc


if __name__ == "__main__":
    sys.exit(main())
