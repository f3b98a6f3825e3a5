"""Shaped structuring elements on one GPU: the morphology kernel's time per step and pass (Handle.kernel_times, the
KERNEL_TIMES brackets), frames/s and the lfd_result bytes, for 64 resident config-3 frames (bench.py's pool) with two
handles taking turns as in bench.py's `value` leg, element by element:

    rect        the default all-ones rectangles (control: the rectangle kernels, untouched by shaped elements)
    cross5      bright dilation cv2 cross 5 x 5           ellipse7x4  bright dilation ellipse 7 x 4 (h x w)
    ellipse9 / ellipse15 / ellipse31 / ellipse41 / ellipse63 / ellipse127
                dim dilation ellipse n x n after the default 3 x 3 erosion

Two builds alternate in the same run, each in its own process (the library is picked by LFD_B200_LIB at import): this
tree's library and a reference build compiled into a temporary directory from --ref-src (a directory holding another
revision's include/ and lfd_b200/csrc/).  An element a build refuses is reported as such.

    python profiles/morph_shapes_bench.py --ref-src DIR [--rounds 2] [--steps 20] [--out FILE]

Prints one JSON line per (round, build, element) and a summary line per element; the device name and power limit are
read in the same run."""
import argparse
import hashlib
import json
import multiprocessing as mp
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np

B = 64
ELEMENTS = ["rect", "cross5", "ellipse7x4", "ellipse9", "ellipse15", "ellipse31", "ellipse41", "ellipse63", "ellipse127"]


def device_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return {"device": name, "power_limit": power}
    except Exception as e:  # noqa: BLE001
        return {"device": None, "power_limit": None, "error": repr(e)}


def element_params(name):
    import cv2
    from lfd_b200.detecttrails import default_params
    pb, pd, _ = default_params()
    if name == "cross5":
        pb["dilateKernel"] = cv2.getStructuringElement(cv2.MORPH_CROSS, (5, 5))
    elif name == "ellipse7x4":
        pb["dilateKernel"] = cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (4, 7))
    elif name.startswith("ellipse"):
        n = int(name[7:])
        pd["dilateKernel"] = cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (n, n))
    return pb, pd


def _gen(job):
    from lfd_b200 import synth
    return synth.make_case(*job)


def make_pool():
    from lfd_b200 import synth
    from lfd_b200.detecttrails import default_params
    from lfd_b200.removestars import star_rects
    _, _, pr = default_params()
    jobs, filters = [], []
    for i in range(B):
        flt = synth.FILTERS[i % 5]
        jobs.append(synth.case_for_frame(2888, 1, flt, 100 + i))
        filters.append(flt)
    with mp.get_context("fork").Pool(min(os.cpu_count() or 1, 32)) as pool:
        made = pool.map(_gen, jobs, chunksize=2)
    rects = [star_rects(m[1], flt, (synth.FRAME_H, synth.FRAME_W), **pr) for m, flt in zip(made, filters)]
    return np.stack([m[0] for m in made]), rects


def worker(args):
    """One build: every element on the same pool; one JSON line each."""
    from lfd_b200 import _lib, synth
    frames, rects = make_pool()
    hs = [_lib.Handle(synth.FRAME_H, synth.FRAME_W, max_batch=B) for _ in range(2)]
    for h in hs:
        h.host_frames[:] = frames
    for name in args.elements:
        out = {"build": args.build, "element": name}
        pb, pd = element_params(name)
        try:
            for h in hs:
                h.set_params(pb, pd)
        except _lib.LfdError as e:
            out["refused"] = str(e)
            print(json.dumps(out), flush=True)
            continue
        for h in hs:
            h.upload(B, rects)

        def loop(steps):
            for k in range(steps):
                if k >= 2:
                    hs[k % 2].wait()
                hs[k % 2].run_resident(B)
            last = None
            for k in range(max(steps - 2, 0), steps):
                last = hs[k % 2].wait_array()
            return last

        loop(3)
        t0 = time.perf_counter()
        res = loop(args.steps)
        out["frames_per_s"] = B * args.steps / (time.perf_counter() - t0)
        out["results_sha256"] = hashlib.sha256(res.tobytes()).hexdigest()
        out["detected"] = int(res["detected"].sum())
        kt = {}
        for _ in range(args.steps // 2):
            hs[0].run_resident(B, flags=_lib.KERNEL_TIMES)
            hs[0].wait()
            for kname, p, ms, _n in hs[0].kernel_times():
                if kname == "k_morph_march":              # the morphology bracket, whichever kernel it holds
                    kt[p] = kt.get(p, 0.0) + ms / (args.steps // 2)
        out["morph_ms_bright"], out["morph_ms_dim"] = kt.get(0, 0.0), kt.get(1, 0.0)
        print(json.dumps(out), flush=True)
    for h in hs:
        h.close()


def build_ref(src, dst):
    from lfd_b200 import _lib
    cmd = ["nvcc"] + _lib.NVCC_FLAGS + [os.path.join(src, "lfd_b200", "csrc", "lfd_b200.cu"), "-o", dst]
    subprocess.run(cmd, check=True)
    return dst


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref-src", help="directory with another revision's include/ and lfd_b200/csrc/")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--elements", nargs="+", default=ELEMENTS)
    ap.add_argument("--out", default=None)
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--build", default="change", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker:
        worker(args)
        return
    from lfd_b200 import _lib
    info = device_info()
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(d)

    with tempfile.TemporaryDirectory() as tmp:
        libs = {"change": _lib.build()}
        if args.ref_src:
            libs["reference"] = build_ref(args.ref_src, os.path.join(tmp, "liblfd_b200_ref.so"))
        rows = []
        for rnd in range(args.rounds):
            for build, path in libs.items():
                env = dict(os.environ, LFD_B200_LIB=path)
                cmd = [sys.executable, os.path.abspath(__file__), "--worker", "--build", build, "--steps", str(args.steps),
                       "--elements"] + args.elements
                p = subprocess.run(cmd, env=env, capture_output=True, text=True, check=True)
                for ln in p.stdout.splitlines():
                    if ln.startswith("{"):
                        d = dict(json.loads(ln), round=rnd, **info)
                        rows.append(d)
                        emit(d)
    for name in args.elements:
        s = {"summary": name, **info}
        for build in libs:
            rs = [r for r in rows if r["element"] == name and r["build"] == build and "refused" not in r]
            if not rs:
                s[build] = "refused"
                continue
            s[build] = {k: [round(r[k], 4) for r in rs] for k in ("morph_ms_bright", "morph_ms_dim", "frames_per_s")}
        hashes = {r["results_sha256"] for r in rows if r["element"] == name and "refused" not in r}
        if all(isinstance(s.get(b), dict) for b in libs) and len(libs) > 1:
            s["results_identical"] = len(hashes) == 1
        emit(s)
    if args.out:
        with open(args.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
