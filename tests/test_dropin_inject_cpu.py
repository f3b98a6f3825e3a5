"""CPU side of injections in a drop-in run (DetectTrails(injections=...)): the injection table's text format against
inject.read_injections, the ordered gather of records that carry injection lines (gloo, world size 2), and the checks
that reject a bad injection specification before anything of its batch is written."""
import io
import math
import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

from lfd_b200 import _lib, inject, synth


def _result(detected, pass_, status, rho, theta):
    r = np.zeros(1, np.dtype(_lib.Result))[0]
    r["detected"], r["pass_"], r["status"], r["rho"], r["theta"] = detected, pass_, status, rho, theta
    return r


def test_write_read_roundtrip_is_bit_exact(tmp_path):
    """Every float32 of a line (end points, sigma, peak, rho, theta) reads back to the same bits: random bit patterns
    over the whole finite range, subnormals, signed zeros and infinities."""
    rng = np.random.default_rng(17)
    bits = rng.integers(0, 2 ** 32, 40000, dtype=np.uint64).astype(np.uint32)
    vals = bits.view(np.float32)
    vals = vals[np.isfinite(vals)]
    special = np.array([0.0, -0.0, np.inf, -np.inf, 1e-45, -1e-45, 1.1754942e-38, 3.4028235e38, 1.0, 0.1], np.float32)
    vals = np.concatenate([special, vals])
    frames, rows, i = [], [], 0
    with open(tmp_path / "injections.txt", "w") as f:
        while i < len(vals):
            n = int(rng.integers(0, 17))
            ts = []
            for _ in range(n):
                v = [float(vals[(i + j) % len(vals)]) for j in range(6)]
                i += 6
                t = {"p0": (v[0], v[1]), "p1": (v[2], v[3]), "sigma": v[4], "peak": v[5]}
                if rng.random() < 0.3:
                    t["profile"] = int(rng.integers(0, 5))
                if rng.random() < 0.3:
                    t["lightcurve"] = int(rng.integers(0, 5))
                ts.append(t)
            r = _result(int(rng.integers(0, 2)), int(rng.integers(-1, 2)), int(rng.integers(0, 8)),
                        vals[i % len(vals)], vals[(i + 1) % len(vals)])
            i += 2
            fr = (int(rng.integers(1, 9000)), int(rng.integers(1, 7)), "ugriz"[int(rng.integers(0, 5))], int(rng.integers(0, 999)))
            k, bd, rec = int(rng.integers(0, 50)), bool(rng.integers(0, 2)), int(rng.integers(-1, max(n, 1)))
            f.write(inject.format_injection(fr, k, bd, ts, r, rec))
            frames.append((fr, k, bd, ts, r, rec))
    tab = inject.read_injections(str(tmp_path / "injections.txt"))
    assert tab.dtype == inject.INJECTION_DTYPE and len(tab) == len(frames)
    for row, (fr, k, bd, ts, r, rec) in zip(tab, frames):
        assert (row["run"], row["camcol"], row["filter"], row["field"]) == fr
        assert row["k"] == k and row["base_detected"] == bd and row["recovered"] == rec
        assert row["detected"] == bool(r["detected"]) and row["pass"] == r["pass_"] and row["status"] == r["status"]
        assert row["rho"].view(np.uint32) == np.float32(r["rho"]).view(np.uint32)
        assert row["theta"].view(np.uint32) == np.float32(r["theta"]).view(np.uint32)
        n = len(ts)
        assert row["ntrails"] == n
        arr = _lib.Handle.trails_array(ts)
        for fld in ("x0", "y0", "x1", "y1", "sigma", "peak"):
            assert np.array_equal(row[fld][:n].view(np.uint32), arr[fld].view(np.uint32)), fld
            assert np.all(np.isnan(row[fld][n:]))
        assert list(row["profile"][:n]) == [t.get("profile", -1) for t in ts]
        assert list(row["lightcurve"][:n]) == [t.get("lightcurve", -1) for t in ts]
        assert np.all(row["profile"][n:] == -1) and np.all(row["lightcurve"][n:] == -1)


def test_nan_sigma_of_a_tabulated_profile_roundtrips(tmp_path):
    t = {"p0": (1.5, 2.0), "p1": (300.25, 400.0), "peak": 2.0, "profile": 0}
    line = inject.format_injection((2888, 3, "r", 12), 0, False, [t], _result(0, -1, 0, 0.0, 0.0), -1)
    assert line == "2888 3 r 12 0 0 0 -1 0 0 0 -1 1 1.5 2 300.25 400 nan 2 0 -1\n"
    (tmp_path / "i.txt").write_text(line)
    row = inject.read_injections(str(tmp_path / "i.txt"))[0]
    assert math.isnan(row["sigma"][0]) and row["profile"][0] == 0 and row["lightcurve"][0] == -1


def _fake_compute(frames):
    """Records like compute_fields with injections: frames with a verdict carry their injection lines (none for some)."""
    out = []
    for (run, camcol, flt, field) in frames:
        if field % 7 == 0:
            out.append(("err", "%d %d %s %d\nboom\n\n" % (run, camcol, flt, field)))
            continue
        rec = ("line", "%d %d %s %d 1 2 3 4\n" % (run, camcol, flt, field)) if field % 3 == 0 else ("none", "")
        if field % 5:
            rec += ("".join("%d %d %s %d %d row\n" % (run, camcol, flt, field, k) for k in range(field % 4)),)
        out.append(rec)
    return out


FRAMES = [(2888, 1, "r", f) for f in range(100, 137)]


def _worker(rank, world, port, tmp):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from lfd_b200.detecttrails import process_fields
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    try:
        res, err, inj = io.StringIO(), io.StringIO(), io.StringIO()
        process_fields(res, err, FRAMES, {"debug": False}, {"debug": False}, {}, batch=4, compute=_fake_compute,
                       injection_results=inj)
        with open(os.path.join(tmp, "out%d.txt" % rank), "w") as f:
            f.write(res.getvalue() + "---\n" + err.getvalue() + "---\n" + inj.getvalue())
    finally:
        dist.destroy_process_group()


def test_gloo_world2_writes_injection_lines_in_frame_order(tmp_path):
    import torch.multiprocessing as mp
    from lfd_b200.detecttrails import process_fields
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    res, err, inj = io.StringIO(), io.StringIO(), io.StringIO()
    prog = str(tmp_path / "progress.txt")
    process_fields(res, err, FRAMES, {"debug": False}, {"debug": False}, {}, batch=4, compute=_fake_compute,
                   distributed=False, progress=prog, injection_results=inj)
    one = res.getvalue() + "---\n" + err.getvalue() + "---\n" + inj.getvalue()
    recs = _fake_compute(FRAMES)
    assert inj.getvalue() == "".join(r[2] for r in recs if len(r) > 2) and inj.getvalue().count("\n") > 20
    assert (tmp_path / "out0.txt").read_text() == one               # rank 0 wrote everything, in sequential order
    assert (tmp_path / "out1.txt").read_text() == "---\n---\n"
    # the progress file lists every frame with its record kind, injection lines or not
    with open(prog) as f:
        assert [ln.split()[4] for ln in f] == [r[0] for r in recs]


@pytest.fixture(scope="module")
def tree(tmp_path_factory):
    import lfd_b200
    root = tmp_path_factory.mktemp("sdss")
    fields = [500, 501, 502, 503]
    t = synth.write_sdss_tree(str(root), 3015, 2, fields, filters=("r",), kinds="sparse", startfield=500, endfield=504)
    lfd_b200.setup(t["bosspath"], t["photoobjpath"], t["photoreduxpath"], str(root))
    return root


def _ok(frame, shape):
    return [[{"p0": (10.0, 20.0), "p1": (1500.0, 1000.0), "sigma": 2.0, "peak": 3.0}]]


@pytest.mark.parametrize("bad", [
    [{"p0": (10.0, 20.0), "p1": (1500.0, 1000.0), "sigma": 2.0, "peak": 3.0}] * 17,
    [{"p0": (math.nan, 20.0), "p1": (1500.0, 1000.0), "sigma": 2.0, "peak": 3.0}],
    [{"p0": (10.0, 20.0), "p1": (1500.0, 1e39), "sigma": 2.0, "peak": 3.0}],            # not finite in float32
    [{"p0": (10.0, 20.0), "p1": (1500.0, 1000.0), "sigma": 2.0, "peak": math.inf}],
    [{"p0": (10.0, 20.0), "p1": (1500.0, 1000.0), "sigma": 0.0, "peak": 3.0}],
    [{"p0": (10.0, 20.0), "p1": (1500.0, 1000.0), "sigma": -1.0, "peak": 3.0}],
    [{"p0": (10.0, 20.0), "p1": (1500.0, 1000.0), "peak": 3.0, "profile": 1}],         # one table in the pool
    [{"p0": (10.0, 20.0), "p1": (1500.0, 1000.0), "sigma": 2.0, "peak": 3.0, "lightcurve": -2}],
    [{"p0": (10.0, 20.0), "p1": (1500.0, 1000.0), "sigma": 2.0, "peak": 3.0, "lightcurve": 1.0}],
    [{"p0": (10.0, 20.0), "p1": (1500.0, 1000.0), "peak": 3.0}],                        # a Gaussian without sigma
    [{"p0": (10.0, 20.0), "sigma": 2.0, "peak": 3.0}],                                  # no p1
    [{"p0": (10.0, 20.0), "p1": (1500.0, 1000.0), "sigma": 2.0, "peak": "bright"}],     # not a number
], ids=["17_trails", "nan", "float32_overflow", "inf_peak", "sigma_0", "sigma_negative", "profile_outside",
        "lightcurve_below", "lightcurve_float", "sigma_missing", "p1_missing", "peak_not_a_number"])
@pytest.mark.parametrize("where", [0, 2])
def test_bad_specification_raises_and_writes_nothing_of_its_batch(tree, tmp_path, bad, where):
    """The bad injection belongs to frame `where` (batch = 2): ValueError out of process(), and none of that batch's
    frames reach results / errors / injections / progress (earlier batches may have been written)."""
    import lfd_b200
    tables = [inject.defocus_profile(6.5, 2.6, 3.5)]

    def inj(frame, shape):
        return [bad] if frame[3] == 500 + where else _ok(frame, shape)

    out = tmp_path / "out"
    out.mkdir()
    dt = lfd_b200.DetectTrails(run=3015, camcol=2, filter="r", savepath=str(out), batch=2, resume=True,
                               injections=inj, injection_tables=tables)
    with pytest.raises(ValueError):
        dt.process()
    done = {int(ln.split()[3]) for ln in open(out / "progress.txt")} if (out / "progress.txt").exists() else set()
    assert done <= set(range(500, 500 + where - where % 2))
    key = " %d\n" % (500 + where)
    assert key not in (out / "errors.txt").read_text() and " %d " % (500 + where) not in (out / "results.txt").read_text()
    assert all(int(ln.split()[3]) in done for ln in open(out / "injections.txt"))


def test_debug_with_injections_raises(tree, tmp_path):
    import lfd_b200
    dt = lfd_b200.DetectTrails(run=3015, camcol=2, filter="r", savepath=str(tmp_path), debug=True, injections=_ok)
    with pytest.raises(ValueError, match="debug"):
        dt.process()
    assert (tmp_path / "results.txt").read_text() == "" and (tmp_path / "errors.txt").read_text() == ""
    assert (tmp_path / "injections.txt").read_text() == ""
