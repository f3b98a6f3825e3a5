"""bench.py's CPU-side pieces (no GPU): workload definitions of BASELINE.json configs 3-5 and the reference arm."""
import json
import os
import subprocess
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    sys.path.insert(0, ROOT)
    import bench
    return bench


def test_workload_params_follow_the_configs():
    bench = _bench()
    import lfd_b200
    pb0, pd0, _ = lfd_b200.default_params()
    name, pb, pd = bench.workload_params(types.SimpleNamespace(workload="config3", hough_method=1.0))
    assert name == "config3-camcol-mix" and pd["houghMethod"] == pd0["houghMethod"] == 20 and pd["dilateKernel"].shape == (9, 9)
    name, pb, pd = bench.workload_params(types.SimpleNamespace(workload="config4", hough_method=2.0))
    assert "config4" in name and pd["dilateKernel"].shape == (15, 15) and pd["houghMethod"] == 2.0
    assert pb["houghMethod"] == pb0["houghMethod"] and pd["erodeKernel"].shape == (3, 3)


def test_config5_grid_and_images():
    bench = _bench()
    cases = bench.c5_cases()
    assert len(cases) == 21 and len(bench.c5_cases(quick=True)) == 4
    assert {c[0] for c in cases} == set(bench.C5_DENSITIES) and {c[1] for c in cases} == set(bench.C5_RHOS)
    assert {round(np.pi / c[2]) for c in cases} == {180, 360, 720, 1440}
    img = bench.c5_image(0.01, 7)
    assert img.shape == (4096, 4096) and img.dtype == np.uint8 and 0.008 < (img != 0).mean() < 0.013
    assert np.array_equal(img, bench.c5_image(0.01, 7))


def test_reference_arm_prints_one_json_line():
    """`bench.py --impl reference` (the CPU arm the driver runs next to ours) needs no GPU; a tiny run must print exactly
    one JSON line with the contract's keys."""
    env = dict(os.environ, OMP_NUM_THREADS="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    assert d["config"]["workload"] == "config3-camcol-mix"


def test_dump_outputs_writes_every_result_field(tmp_path):
    """--dump-outputs: one float64 .npy per lfd_result field of the step's frames, frames first, values exact."""
    bench = _bench()
    from lfd_b200 import _lib
    rs = [_lib.Result(), _lib.Result()]
    rs[0].detected, rs[0].pass_, rs[0].theta = 1, 1, np.float32(0.1)
    rs[1].rect_detection[1] = 7
    rs[1].top_box[1][15][0] = np.float32(-2.5)
    bench.dump_arrays(str(tmp_path / "out"), bench.result_arrays("resident", [bytes(r) for r in rs]))
    names = sorted(p.name for p in (tmp_path / "out").iterdir())
    assert names == sorted("resident_%s.npy" % f.rstrip("_") for f, _t in _lib.Result._fields_)
    load = lambda n: np.load(tmp_path / "out" / ("resident_%s.npy" % n))   # noqa: E731
    assert all(np.load(tmp_path / "out" / n).dtype == np.float64 for n in names)
    assert load("detected").tolist() == [1, 0] and load("pass").tolist() == [1, 0]
    assert load("theta")[0] == np.float32(0.1) and load("rect_detection").tolist() == [[0, 0], [0, 7]]
    assert load("top_box").shape == (2, 2, 16, 2) and load("top_box")[1, 1, 15, 0] == -2.5


def test_roofline_names_the_time_dominant_kernel():
    """build_roofline: the kernel with the most bracketed time per step (all launches of the function together) is the one
    named, whatever stage it belongs to; the streaming-stage kernel is kept beside it."""
    import bench
    N = 1489 * 2048

    def row(k, p, ms, nl, alg=None, des=None):
        e = {"kernel": k, "pass": p, "ms_per_step": ms, "launches_per_step": nl}
        if alg is not None:
            e.update(alg_bytes_per_step=alg, design_bytes_per_step=des)
        return e

    kt = [row("k_prep", "both", 0.23, 1, 64 * 6 * N, 64 * 6 * N),
          row("k_morph_march", "bright", 0.19, 2, 64 * 4 * N, 64 * (2 * N + N // 8)), row("k_morph_march", "dim", 0.46, 2, 56 * 6 * N, 56 * (2 * N + N // 8)),
          row("k_nms_march", "bright", 0.31, 2, 64 * 2 * N, 64 * (N + N // 4)), row("k_nms_march", "dim", 0.33, 2, 56 * 2 * N, 56 * (N + N // 4)),
          row("k_ccl_band(fg)", "bright", 0.23, 2, 64 * 5 * N, 64 * 700000), row("k_ccl_band(fg)", "dim", 0.30, 2, 56 * 5 * N, 56 * 700000),
          row("k_ccl_band(bg)", "bright", 0.19, 2, 64 * 4 * N, 64 * 700000), row("k_ccl_band(bg)", "dim", 0.24, 2, 56 * 4 * N, 56 * 700000),
          row("k_rects_warp", "bright", 0.2, 2), row("k_hough_vote", "dim", 0.24, 2)]
    stage_ms = [("bright:lut+morph", 0.1), ("dim:lut+morph(+x)", 0.2), ("bright:sobel+nms", 0.15), ("dim:sobel+nms", 0.19)]
    measured = {"k_ccl_band": 147.4e6, "k_morph_march": 685.8e6, "k_hough_vote": 4.7e6}
    r, table = bench.build_roofline([dict(e) for e in kt], 6553.9, "measured", measured, "profiles/x.json", stage_ms, 5, 1.9)
    assert r["kernel"] == "k_ccl_band" and abs(r["ms_per_step"] - 0.96) < 1e-9 and r["launches_per_step"] == 8
    assert r["frac"] == r["frac_design_bytes"] and r["frac"] < 0.05 < r["frac_survey_bytes"]        # run-based labelling: design bytes
    assert abs(r["achieved"] - r["frac"] * r["peak"]) < 1e-6 * r["peak"]
    assert r["traffic"] == 147.4e6 / 8
    assert r["hbm_stage"]["kernel"] == "k_morph_march" and "alone" in r["hbm_stage"]
    assert abs(r["hbm_stage"]["alone"]["ms_per_step"] - 0.3) < 1e-9
    assert list(r["all_kernel_ms_per_step"])[0] == "k_ccl_band"
    assert [e["ms_per_step"] for e in table] == sorted((e["ms_per_step"] for e in table), reverse=True)
    # a streaming kernel on top: the survey's bytes are `frac`
    kt2 = [dict(e) for e in kt if not e["kernel"].startswith("k_ccl_band")]
    r2, _ = bench.build_roofline(kt2, 6553.9, "measured", measured, "profiles/x.json", stage_ms, 5, 1.9)
    assert r2["kernel"] == "k_morph_march" and r2["frac"] == r2["frac_survey_bytes"] and r2["alone"]["frac"] > r2["frac"]
    # a kernel the survey has no byte figure for: measured DRAM bytes, flagged
    kt3 = kt2 + [row("k_hough_vote", "bright", 2.0, 2)]
    r3, _ = bench.build_roofline(kt3, 6553.9, "measured", measured, "profiles/x.json", stage_ms, 5, 1.9)
    assert r3["kernel"] == "k_hough_vote" and "measured DRAM" in r3["bytes_model"] and r3["frac"] < 0.01
    r4, _ = bench.build_roofline(kt3, 6553.9, "measured", {}, None, stage_ms, 5, 1.9)
    assert r4["kernel"] == "k_hough_vote" and r4["frac"] is None and r4["achieved"] is None
