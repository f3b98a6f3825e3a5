"""Injection-campaign throughput on one GPU: 64 config-3 bases (sparse and dense mix, synth.case_for_frame) resident on
the device and a grid of single-trail injections (angles incl. 0 and 90 +- 1 degrees, four widths, six peaks, four
lengths), run through lfd_submit_injected with one handle and with two alternating handles; k_inject's event time per
64-slot step against the HBM copy peak; and, for comparison, the same injections rendered on the host with
oracle/inject_ref.py::render_trails (one host thread) and sent through lfd_submit.  The host path renders ~10 ms a
frame, so it runs on the first --host-steps steps of the grid only (stated in its line; 0 skips it).

--shape picks the trail cross-sections, on the same bases and the same geometry grid: ``gaussian`` (synth's Gaussian,
lfd_submit_injected), ``donut`` (lfd_b200.inject.defocus_profile with r_outer 4, 6.67, 9.33, 12 px in place of the four
FWHMs, r_inner = 0.4 r_outer, seeing FWHM 3.5 px; lfd_submit_injected_shaped) and ``donut_lightcurve`` (the same with a
64-sample rise-and-fade light curve).  Several shapes alternate within each round of handle counts.

    python profiles/inject_bench.py [--injections 20480] [--host-steps 8] [--shape gaussian donut ...] [--out DIR]

Prints one JSON line per measurement (and writes them to DIR/inject_bench.jsonl with --out).  The device name and
power limit are read in the same run."""
import argparse
import itertools
import json
import math
import multiprocessing as mp
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np

from lfd_b200 import _lib, synth

B = 64
H, W = synth.FRAME_H, synth.FRAME_W


def device_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return {"device": name, "power_limit": power}
    except Exception as e:  # noqa: BLE001
        return {"device": None, "power_limit": None, "error": repr(e)}


def _gen(job):
    return synth.make_case(*job)


def make_bases():
    from lfd_b200.removestars import star_rects
    from lfd_b200.detecttrails import default_params
    _, _, pr = default_params()
    jobs, filters = [], []
    for i in range(B):
        flt = synth.FILTERS[i % 5]
        jobs.append(synth.case_for_frame(2888, 6, flt, 500 + i))
        filters.append(flt)
    with mp.get_context("fork").Pool(min(os.cpu_count() or 1, 32)) as pool:
        made = pool.map(_gen, jobs, chunksize=2)
    frames = np.stack([m[0] for m in made])
    rects = [star_rects(m[1], flt, (H, W), **{k: v for k, v in pr.items()}) for m, flt in zip(made, filters)]
    return frames, rects, [j[0] for j in jobs]


FWHM = (2.0, 4.0, 8.0, 15.0)
R_OUTER = (4.0, 20.0 / 3.0, 28.0 / 3.0, 12.0)     # the donut that replaces FWHM[k]
COMBOS = list(itertools.product((0.0, 1.0, 179.0, 89.0, 90.0, 91.0, 30.0, 45.0, 60.0, 120.0, 135.0, 150.0), FWHM,
                                (0.1, 0.3, 1.0, 3.0, 10.0, 50.0), (200.0, 600.0, 1200.0, 2400.0)))


def make_grid(n, seed=2026):
    """n single-trail injections: every combination of 12 angles, 4 FWHMs, 6 peaks and 4 lengths, repeated with random
    centres (middle half of the frame) and random bases."""
    rng = np.random.default_rng(seed)
    combos = COMBOS
    out = []
    for i in range(n):
        ang, fw, pk, L = combos[i % len(combos)]
        a = math.radians(ang)
        cx, cy = rng.uniform(0.25 * W, 0.75 * W), rng.uniform(0.25 * H, 0.75 * H)
        out.append((int(rng.integers(0, B)), [{"p0": (cx - L / 2 * math.cos(a), cy - L / 2 * math.sin(a)),
                                               "p1": (cx + L / 2 * math.cos(a), cy + L / 2 * math.sin(a)),
                                               "sigma": fw / 2.3548, "peak": pk}]))
    return out


def shape_tables():
    """The donut profiles (table k replaces FWHM[k]) and, last, the rise-and-fade light curve."""
    from lfd_b200.inject import defocus_profile
    s = np.linspace(0.0, 1.0, 64)
    rise_fade = np.where(s < 0.3, (s / 0.3) ** 2, np.exp(-(s - 0.3) / 0.35)).astype(np.float32)
    return [defocus_profile(r, 0.4 * r, 3.5) for r in R_OUTER] + [(0.0, 1.0, rise_fade)]


def shaped_grid(grid, shape):
    """The grid with the trails of `shape`: the same end points and peaks, the Gaussian of FWHM[k] replaced by donut k."""
    if shape == "gaussian":
        return grid
    out = []
    for i, (b, (t,)) in enumerate(grid):
        t = dict(t, profile=FWHM.index(COMBOS[i % len(COMBOS)][1]))
        del t["sigma"]
        if shape == "donut_lightcurve":
            t["lightcurve"] = len(R_OUTER)
        out.append((b, [t]))
    return out


def hbm_peak():
    """(GB/s, source): MEASURED_PEAKS.json's hbm_gbs when present, else a device-to-device copy measured here."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    import torch
    a = torch.empty(1 << 29, dtype=torch.float32, device="cuda")      # 2 GiB, far beyond the L2
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 20
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    gbs = 2 * a.numel() * 4 * reps / (e0.elapsed_time(e1) * 1e6)
    del a, b
    return gbs, "device-to-device copy of 2 GiB measured in this run (torch copy_, read + write bytes)"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--injections", type=int, default=20480)
    ap.add_argument("--host-steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shape", nargs="+", default=["gaussian"], choices=["gaussian", "donut", "donut_lightcurve"])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from lfd_b200.detecttrails import default_params
    from oracle.inject_ref import render_trails

    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(d)

    info = device_info()
    frames, rects, kinds = make_bases()
    grid = make_grid(args.injections)
    steps = [grid[i:i + B] for i in range(0, len(grid), B)]
    pb, pd, _ = default_params()
    hs = [_lib.Handle(H, W, max_batch=B) for _ in range(2)]
    tables = shape_tables()
    for h in hs:
        h.set_params(pb, pd)
        h.set_base(frames, rects)
        h.set_trail_tables(tables)
    common = dict(info, bases=B, base_kinds={k: kinds.count(k) for k in sorted(set(kinds))}, batch=B,
                  frame=[H, W], injections=len(grid))

    def run_device(nh, which):
        """All steps, `nh` handles taking turns; returns (seconds, [k_inject ms per step], detections)."""
        kms, ndet = [], 0

        def submit(k):
            s = which[k]
            hs[k % nh].submit_injected([b for b, _ in s], [ts for _, ts in s])

        def collect(k):
            nonlocal ndet
            h = hs[k % nh]
            r = h.wait_array()
            ndet += int(r["detected"].sum())
            kms.append(h.kernel_times()[-1][2])

        t0 = time.perf_counter()
        submit(0)
        for k in range(1, len(which)):
            if nh == 1:
                collect(k - 1)
            submit(k)
            if nh == 2:
                collect(k - 1)
        collect(len(which) - 1)
        return time.perf_counter() - t0, kms, ndet

    # k_inject against the HBM peak: 8 N bytes per slot (read the base, write the batch slot).  With one handle the
    # kernel runs alone; with two it overlaps the other handle's passes, so its event time includes their contention.
    peak, src = hbm_peak()
    bytes_step = 8 * H * W * B
    shaped = {}
    for sh in args.shape:
        g = shaped_grid(grid, sh)
        shaped[sh] = [g[i:i + B] for i in range(0, len(g), B)]
    for sh in args.shape:
        run_device(2, shaped[sh][:args.warmup])
    for nh, sh in itertools.product((1, 2, 1, 2), args.shape):
        dt, kms, ndet = run_device(nh, shaped[sh])
        ms = float(np.median(kms))
        step_ms = 1e3 * dt / len(steps)
        emit(dict(common, metric="injections/s (lfd_submit_injected, bases resident)", handles=nh, shape=sh,
                  value=len(grid) / dt, seconds=dt, steps=len(steps), detections=ndet, step_ms=step_ms,
                  k_inject={"ms_median": ms, "ms_min": float(np.min(kms)), "ms_max": float(np.max(kms)),
                            "bytes_per_step": bytes_step, "gbs": bytes_step / (ms * 1e6), "hbm_peak_gbs": peak,
                            "hbm_peak_source": src, "frac_of_hbm_peak": bytes_step / (ms * 1e6) / peak,
                            "share_of_step": ms / step_ms}))
    # the same injections rendered on the host and sent over PCIe (two handles double-buffered)
    hsteps = steps[:args.host_steps]

    def host_stage(k):
        h = hs[k & 1]
        for j, (b, ts) in enumerate(hsteps[k]):
            np.copyto(h.host_frames[j], frames[b])
            render_trails(h.host_frames[j], ts)
        h.submit(len(hsteps[k]), [rects[b] for b, _ in hsteps[k]])

    if hsteps:
        host_stage(0)
        hs[0].wait()
        t0 = time.perf_counter()
        host_stage(0)
        for k in range(1, len(hsteps)):
            host_stage(k)
            hs[(k - 1) & 1].wait()
        hs[(len(hsteps) - 1) & 1].wait()
        dt = time.perf_counter() - t0
        n = sum(len(s) for s in hsteps)
        emit(dict(common, metric="injections/s (render_trails on the host, one thread, + lfd_submit)", handles=2,
                  shape="gaussian", value=n / dt, seconds=dt, injections=n, note="first %d steps of the grid" % len(hsteps)))
    for h in hs:
        h.close()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "inject_bench.jsonl"), "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
