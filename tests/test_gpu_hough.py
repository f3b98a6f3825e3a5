"""The Hough stage, exactly: k_hough_compact, k_hough_vote on every path, k_hough_peaks, k_hough_topk, k_hough_sort,
k_check_theta and k_finalize (lfd_b200/csrc/k_hough.cuh, lfd_b200.cu).

k_hough_vote takes one of these paths per (non-zero 32-pixel mask word, angle), with r1 / r2 the bins of the word's
first and last set pixel:
  single             r1 == r2: one shared-memory atomic of weight popc;
  two                |r2 - r1| == 1 and popc > 4: the boundary is located by last_with, two atomics;
  three_mid_set      |r2 - r1| == 2, popc > 4, the middle bin rm holds set pixels: three atomics;
  three_mid_empty    the same with no set pixel in the middle bin (the `if (c2)` branch): two atomics;
  three_mid_skipped  |r2 - r1| == 2 but the bin after r1 is r2 (rm == r2): two atomics;
  pixel_coarse       0 < |r2 - r1| <= 2 with popc <= 4: every pixel votes on its own;
  pixel_fine         |r2 - r1| > 2: every pixel votes on its own.
last_with predicts the boundary from the real-valued line, clamps the prediction into the interval, probes it and its
neighbour and bisects what is left; each boundary is classed by how far the prediction lands from the answer
(predicted, off_by_one, off_by_more).  vote_paths() restates all of it in NumPy float32 (separate roundings,
round-half-even, __frcp_rn as a correctly rounded float32 division, the magic conversions with int32 wrap-around), and
restates device counter 13 (hough_smem_atomics), which depends only on these paths.  setup() and nchunks() restate the
CTA-level choices of hough_setup and k_hough_vote (angles per CTA, per, privatised copies); their constants are read
from the CUDA sources, so changing one fails a test instead of quietly retiring a case.

three_mid_skipped cannot occur: with popc > 4 the word spans at least 4 pixels, two bin boundaries inside that span
need |cos / rho| below about 0.5 per pixel, while skipping the middle bin in one pixel step needs it near 1.  The
coverage test asserts it stays at zero; reaching it would be a finding.

The magic conversions (hough_magic_ok) hold for every frame and rho hough_setup accepts (apc >= 1 bounds numrho by
24 573, so (W + H) / rho stays below about 12 300, and lfd_hough_lines caps W at 65 535 * 32 < 2^23), so the
k_hough_vote<false> instantiation is unreachable; test_magic_path_covers_every_accepted_setup pins that."""
import math
import os
import re

import numpy as np
import pytest

from oracle import cv_restate as cr
from oracle import ref_pipeline as rp

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "lfd_b200", "csrc")
F32 = np.float32


def _read(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _constants():
    kh, cu = _read("k_hough.cuh"), _read("lfd_b200.cu")
    c = {k: int(re.search(r"#define\s+%s\s+(\d+)" % k, kh).group(1)) for k in ("HOUGH_THREADS", "HOUGH_MIN_SEGS")}
    c["SMEM_BUDGET"] = int(re.search(r"smem_budget\s*=\s*(\d+)\s*\*\s*1024\s*;", cu).group(1)) * 1024
    c["BY_PAR"] = int(re.search(r"by_par\s*=\s*\((\d+)\s*\+", kh).group(1))
    grids = set(re.findall(r"k_hough_vote<(?:true|false)><<<dim3\((\d+),", cu))
    assert len(grids) == 1, grids
    c["GRID_X"] = int(grids.pop())
    c["MAGIC_W"], c["MAGIC_RHO"] = (float(v) for v in re.search(
        r"hough_magic_ok\(int H, int W, float rho\)\s*\{\s*return W < \(1 << (\d+)\) && \(double\)\(W \+ H\) / rho < ([\d.]+);",
        kh).groups())
    return c


K = _constants()


# ---- restatement --------------------------------------------------------------------------------------------------
def dims(H, W, rho, theta):
    """hough_dims_host: float theta and rho, float (na - 1) * theta, float division for numrho, lrint."""
    th, r = F32(theta), F32(rho)
    na = int(math.floor(math.pi / float(th))) + 1
    if na > 1 and abs(math.pi - float(F32(na - 1) * th)) < float(th) / 2:
        na -= 1
    return na, int(np.rint(F32(2 * (W + H) + 1) / r))


def tables(na, rho, theta):
    """OpenCV's tables: float32 accumulated angle, sin / cos in double times the float32 1 / rho, rounded to float."""
    irho, th, ang = F32(1) / F32(rho), F32(theta), F32(0)
    ts, tc = np.empty(na, F32), np.empty(na, F32)
    for n in range(na):
        ts[n] = F32(math.sin(float(ang)) * float(irho))
        tc[n] = F32(math.cos(float(ang)) * float(irho))
        ang = F32(ang + th)
    return ts, tc


def _next_pow2(v):
    p = 1
    while p < v:
        p <<= 1
    return p


def setup(H, W, rho, theta):
    """hough_setup: dict(err, na, nr, RS, RSS, apc, ngroups, per); err is "arg" or "unsupported" where it refuses."""
    na, nr = dims(H, W, rho, theta)
    if na < 1 or nr < 1 or na * nr > 2.0e8:
        return {"err": "arg"}
    RS = nr + 2
    RSS = RS | 1
    apc = min(K["SMEM_BUDGET"] // (RSS * 4), 32)
    if apc < 1:
        return {"err": "unsupported"}
    if apc < 32:
        apc = 1 << (apc.bit_length() - 1)
    if apc > na:
        apc = _next_pow2(na) if na < 32 else 32
    return {"err": None, "na": na, "nr": nr, "RS": RS, "RSS": RSS, "apc": apc, "ngroups": -(-na // apc),
            "per": 1 if apc >= 32 else 32 // apc, "rho": rho, "theta": theta}


def nchunks(cfg, nseg, nnz, gz=1):
    """k_hough_vote's privatised copies of an (image, angle group) and the term that bound them."""
    by_seg = min(K["GRID_X"], max(1, -(-nseg // K["HOUGH_MIN_SEGS"])))
    by_votes = max(1, nnz // (8 * cfg["RSS"]))
    by_par = -(-K["BY_PAR"] // (cfg["ngroups"] * gz))
    n = min(by_seg, max(by_votes, by_par))
    return n, ("seg" if by_seg <= max(by_votes, by_par) else "votes" if by_votes >= by_par else "par")


def R(x, c, ys):
    return np.rint(np.asarray(x).astype(F32) * c + ys).astype(np.int64)


def _last_with(allr, lo_in, hi_in, rr):
    """largest x in [lo_in, hi_in) with R(x) == rr (R is monotone in x)"""
    xs = np.arange(32)
    eq = (allr == rr[:, None]) & (xs >= lo_in[:, None]) & (xs < hi_in[:, None])
    return 31 - np.argmax(eq[:, ::-1], 1)


def _prediction(lo_in, hi_in, rr, half, ys, inv_c, x0f, answer):
    """last_with's clamped prediction (magic rint of ((rr + half) - ys) * inv_c - x0) against the answer:
    counts of (exact, off by one, off by more)."""
    xg = ((rr.astype(F32) + half) - ys) * inv_c - x0f
    with np.errstate(over="ignore", invalid="ignore"):
        g = (xg + F32(12582912.0)).view(np.int32).astype(np.int64) - 0x4B400000
    g = ((g + (1 << 31)) % (1 << 32)) - (1 << 31)
    g = np.minimum(np.maximum(g, lo_in), hi_in - 1)
    return np.bincount(np.minimum(np.abs(g - answer), 2), minlength=3)


CLASSES = ("single", "two", "three_mid_set", "three_mid_empty", "three_mid_skipped", "pixel_coarse", "pixel_fine")
PRED = ("predicted", "off_by_one", "off_by_more")


def _words(img):
    H, W = img.shape
    WW = (W + 31) // 32
    pad = np.zeros((H, WW * 32), bool)
    pad[:, :W] = img != 0
    bits = pad.reshape(H, WW, 32)
    ys, ws = np.nonzero(bits.any(2))
    return ys, ws, bits[ys, ws]


def vote_paths(img, cfg):
    """Per-class (word, angle) counts, boundary prediction classes, the boundary offsets inside the word (set of lo),
    crossings at |cos| < 1e-3 and the restated counter 13 ("atomics")."""
    ys_i, ws, wb = _words(img)
    out = dict.fromkeys(CLASSES + PRED, 0)
    out.update(near90=0, atomics=0, nseg=len(ys_i), nnz=int(wb.sum()), offsets=set())
    if not len(ys_i):
        return out
    pc = wb.sum(1)
    fb, lb = wb.argmax(1), 31 - wb[:, ::-1].argmax(1)
    x0 = ws.astype(np.int64) * 32
    x0f, yf = x0.astype(F32), ys_i.astype(F32)
    ts, tc = tables(cfg["na"], cfg["rho"], cfg["theta"])
    xs = np.arange(32)
    for n in range(cfg["na"]):
        c, s = tc[n], ts[n]
        ys = yf * s
        r1, r2 = R(x0 + fb, c, ys), R(x0 + lb, c, ys)
        d = np.abs(r2 - r1)
        coarse, fine = (d > 0) & (d <= 2) & (pc <= 4), d > 2
        out["single"] += int((d == 0).sum())
        out["pixel_coarse"] += int(coarse.sum())
        out["pixel_fine"] += int(fine.sum())
        out["atomics"] += int((d == 0).sum()) + int(pc[coarse | fine].sum())
        if abs(float(c)) < 1e-3:
            out["near90"] += int((d > 0).sum())
        k = np.nonzero((d > 0) & (d <= 2) & (pc > 4))[0]
        if not len(k):
            continue
        inv_c = F32(1) / c
        half = np.where(r2[k] > r1[k], F32(0.5), F32(-0.5)).astype(F32)
        allr = R(x0[k, None] + xs[None, :], c, ys[k, None])
        lo = _last_with(allr, fb[k], lb[k], r1[k])
        for p, v in zip(PRED, _prediction(fb[k], lb[k], r1[k], half, ys[k], inv_c, x0f[k], lo)):
            out[p] += int(v)
        out["offsets"].update(lo.tolist())
        hi = lo + 1
        rm = allr[np.arange(len(k)), hi]
        two = d[k] == 1
        skip = (d[k] == 2) & (rm == r2[k])
        t = np.nonzero((d[k] == 2) & (rm != r2[k]))[0]
        out["two"] += int(two.sum())
        out["three_mid_skipped"] += int(skip.sum())
        out["atomics"] += 2 * int((two | skip).sum())
        if len(t):
            lo2 = _last_with(allr[t], hi[t], lb[k][t], rm[t])
            for p, v in zip(PRED, _prediction(hi[t], lb[k][t], rm[t], half[t], ys[k][t], inv_c, x0f[k][t], lo2)):
                out[p] += int(v)
            out["offsets"].update(lo2.tolist())
            c2 = ((xs[None, :] >= hi[t, None]) & (xs[None, :] <= lo2[:, None]) & wb[k][t]).sum(1)
            out["three_mid_set"] += int((c2 > 0).sum())
            out["three_mid_empty"] += int((c2 == 0).sum())
            out["atomics"] += 2 * len(t) + int((c2 > 0).sum())
    return out


def ties(img, cfg, angles):
    """(pixel, angle) pairs at the given angle indices whose x * c + y * s is exactly k + 0.5 (round-half-even)."""
    ys, xs = np.nonzero(img)
    ts, tc = tables(cfg["na"], cfg["rho"], cfg["theta"])
    n = 0
    for a in angles:
        v = xs.astype(F32) * tc[a] + ys.astype(F32) * ts[a]
        n += int((v - np.floor(v) == F32(0.5)).sum())
    return n


PEAK_KINDS = ("eq_left", "eq_right", "eq_up", "eq_down", "row_first", "row_last", "col_first", "col_last")


def peak_kinds(acc, threshold):
    """Cells where one of k_hough_peaks' four comparisons is decided by equality while the other three pass, and peaks
    in the first / last angle row and rho column."""
    A = acc.astype(np.int64)
    v = A[1:-1, 1:-1]
    left, right, up, down = A[1:-1, :-2], A[1:-1, 2:], A[:-2, 1:-1], A[2:, 1:-1]
    big = v > threshold
    peak = big & (v > left) & (v >= right) & (v > up) & (v >= down)
    out = {"eq_left": big & (v == left) & (v >= right) & (v > up) & (v >= down),
           "eq_right": big & (v > left) & (v == right) & (v > up) & (v >= down),
           "eq_up": big & (v > left) & (v >= right) & (v == up) & (v >= down),
           "eq_down": big & (v > left) & (v >= right) & (v > up) & (v == down)}
    out = {k: int(m.sum()) for k, m in out.items()}
    out.update(row_first=int(peak[0].sum()), row_last=int(peak[-1].sum()), col_first=int(peak[:, 0].sum()),
               col_last=int(peak[:, -1].sum()))
    return out


# ---- images ---------------------------------------------------------------------------------------------------------
def _random_words(rng, H, W, nwords, lo=5, hi=32):
    """nwords distinct mask words with lo..hi set pixels at random places (the last word of a row clipped at W)."""
    img = np.zeros((H, W), np.uint8)
    WW = (W + 31) // 32
    for i in rng.choice(H * WW, size=min(nwords, H * WW), replace=False):
        y, w = divmod(int(i), WW)
        bits = rng.choice(32, size=int(rng.integers(lo, hi + 1)), replace=False)
        xs = w * 32 + bits
        img[y, xs[xs < W]] = int(rng.integers(1, 256))
    return img


def img_boundary_words(H=256, W=1024, seed=1):
    """Words with 5..32 set pixels everywhere in the frame, so that at every rho some boundary falls at every offset
    inside a word, plus short words (popc <= 4) that cross a boundary at coarse rho."""
    rng = np.random.default_rng(seed)
    img = _random_words(rng, H, W, 1500)
    img |= _random_words(rng, H, W, 300, 1, 4)
    return img


def img_ties(H=64, W=96):
    """Odd x on row 0 (x * 0.5 = k + 0.5 at rho = 2, theta = 0) and full words on odd rows, where tabSin[90] = 0.5 at
    rho = 2 puts ys on k + 0.5 and the tiny non-zero tabCos[90] moves the word's later pixels off it: round-half-even
    decides both."""
    img = np.zeros((H, W), np.uint8)
    img[0, 1::2] = 255
    img[1::4, :64] = 255
    return img


def img_near90(H=1200, W=640):
    """Full words on every row: rows where y * tabSin lies just above k + 0.5 cross a bin a few pixels into the word at
    the angles next to 90 degrees, where the prediction (inv_c ~ 1e6) is clamped and bisection finishes."""
    img = np.zeros((H, W), np.uint8)
    img[:, :96] = 255
    img[::7, 96:W:2] = 255
    return img


def img_edges(H, W):
    """Pixels at x = 0, y = 0, x = W - 1 and y = H - 1, and in the corners."""
    img = np.zeros((H, W), np.uint8)
    img[0, :: max(1, W // 7)] = 255
    img[H - 1, :: max(1, W // 5)] = 255
    img[:: max(1, H // 7), 0] = 255
    img[:: max(1, H // 3), W - 1] = 255
    img[0, 0] = img[H - 1, W - 1] = img[0, W - 1] = img[H - 1, 0] = 255
    return img


def img_sort(votes, gap=2, H=4):
    """theta = 3.0 keeps one angle (0): a column x = gap * i with votes[i] set pixels is an isolated accumulator cell,
    so there is exactly one peak per column and the peaks' order is decided by votes and then by index."""
    W = gap * len(votes) + 1
    img = np.zeros((H, W), np.uint8)
    for i, v in enumerate(votes):
        img[:v, gap * i] = 255
    return img


def standalone_cases():
    """(name, image, rho, theta, threshold) of the standalone lfd_hough_lines tests."""
    out = []
    bw = img_boundary_words()
    for rho in (20, 5, 2, 1, 0.5):
        out.append(("boundary_words", bw, rho, np.pi / 180, 1))
    out.append(("ties", img_ties(), 2, np.pi / 180, 1))
    for rho in (20, 5, 2, 1):
        out.append(("near90", img_near90(), rho, np.pi / 180, 1))
    for H, W in ((37, 33), (40, 63), (1, 1), (1, 95), (70, 1), (5, 31)):
        for rho in (1, 3, 20):
            out.append(("edges", img_edges(H, W), rho, np.pi / 180, 0))
    big = np.zeros((65535, 32), np.uint8)
    big[::4093, :] = 255
    big[65535 - 1, [0, 31]] = 255
    big[32768:32800, 5:12] = 255
    out.append(("tall", big, 20, np.pi / 180, 1))
    wide = np.zeros((1, 65535 * 32), np.uint8)
    wide[0, ::4099] = 255
    wide[0, -40:] = 255
    out.append(("wide", wide, 200, np.pi / 180, 1))
    # apc 32 .. 1 and per 1 .. 32 on 45 words (not a multiple of any per) and on 7 words (fewer than per)
    rng = np.random.default_rng(5)
    few, fewer = _random_words(rng, 97, 300, 45), _random_words(rng, 97, 300, 7)
    for theta in (np.pi / 180, np.pi / 360, 0.1, 0.5, 1.0, 3.0):
        for apc in (32, 16, 8, 4, 2, 1):
            rho = (2 * (97 + 300) + 1) / (0.75 * (K["SMEM_BUDGET"] // 4) / apc)
            out.append(("apc", few if apc % 2 else fewer if apc == 4 else few, rho, theta, 1))
    # privatised copies: one owner (few segments), many by segments, bound by parallelism and by votes per cell
    dense = np.zeros((600, 1000), np.uint8)
    dense[:, :] = (np.random.default_rng(6).random((600, 1000)) < 0.9) * 255
    out.append(("nchunks_votes", dense, 0.4, np.pi / 180, 1))
    out.append(("nchunks_par", _random_words(rng, 600, 1000, 3000), 0.5, np.pi / 180, 1))
    out.append(("nchunks_seg", _random_words(rng, 300, 640, 2000), 20, np.pi / 180, 1))
    out.append(("nchunks_single", _random_words(rng, 300, 640, 400), 20, np.pi / 180, 1))
    out.append(("nchunks_seg_min", _random_words(rng, 300, 640, K["HOUGH_MIN_SEGS"]), 20, np.pi / 180, 1))
    out.append(("nchunks_seg_min1", _random_words(rng, 300, 640, K["HOUGH_MIN_SEGS"] + 1), 3, np.pi / 180, 1))
    return [c for c in out if setup(c[1].shape[0], c[1].shape[1], c[2], c[3])["err"] is None]


def _coverage(cases):
    tot = dict.fromkeys(CLASSES + PRED, 0)
    regimes, apcs, pers, rs_par, near90, offsets = set(), set(), set(), set(), 0, {}
    for name, img, rho, theta, thr in cases:
        cfg = setup(img.shape[0], img.shape[1], rho, theta)
        o = vote_paths(img, cfg)
        for k in tot:
            tot[k] += o[k]
        near90 += o["near90"]
        offsets.setdefault(rho, set()).update(o["offsets"])
        n, reg = nchunks(cfg, o["nseg"], o["nnz"])
        regimes.add((reg, "single" if n == 1 else "atomic"))
        apcs.add(cfg["apc"])
        pers.add((cfg["per"], o["nseg"] < cfg["per"], o["nseg"] % cfg["per"] != 0))
        rs_par.add(cfg["RS"] % 2)
    return tot, regimes, apcs, pers, rs_par, near90, offsets


def img_peaks():
    """Small images whose accumulators hold plateaus in both directions and peaks next to the zero padding."""
    out = [img_edges(5, 31), img_edges(1, 1), img_sort([1, 1, 2, 2, 3, 1, 3]), img_ties()]
    tiny = np.zeros((3, 3), np.uint8)
    tiny[1, :] = 255
    out.append(tiny)
    return out


# ---- CPU tests ------------------------------------------------------------------------------------------------------
def test_tables_and_dims_match_oracle():
    """dims() and tables() equal oracle/cv_restate's orc_hough_dims / orc_hough_tables bit for bit (the oracle is pinned
    to cv2.HoughLines in tests/test_oracle_cv.py)."""
    import ctypes
    for H, W in ((1, 1), (65535, 32), (1, 65535 * 32), (97, 300), (1489, 2048)):
        for rho in (0.043, 0.4, 0.5, 1, 1.38, 2, 3, 5, 20, 200):
            for theta in (np.pi / 180, np.pi / 360, 0.1, 0.5, 1.0, 3.0, 1e-5):
                na, nr = dims(H, W, rho, theta)
                assert (na, nr) == cr.hough_dims(H, W, rho, theta), (H, W, rho, theta)
                if na > 4096:
                    continue
                a, b = np.empty(na, F32), np.empty(na, F32)
                cr.lib().orc_hough_tables(na, ctypes.c_double(rho), ctypes.c_double(theta), cr._p(a), cr._p(b))
                ts, tc = tables(na, rho, theta)
                assert np.array_equal(a.view(np.uint32), ts.view(np.uint32)) and np.array_equal(b.view(np.uint32), tc.view(np.uint32))


def test_magic_path_covers_every_accepted_setup():
    """hough_magic_ok holds wherever hough_setup accepts a frame: at every rho, the largest W + H it accepts keeps
    (W + H) / rho under the magic bound, and lfd_hough_lines' widest frame stays under 2^MAGIC_W.  So k_hough_vote<false>
    is unreachable."""
    assert 65535 * 32 < 2 ** K["MAGIC_W"]
    for rho in np.geomspace(0.01, 2000, 400):
        s = int(math.floor((24573.5 * float(F32(rho)) - 1) / 2)) + 3
        while s > 2 and setup(1, s - 1, rho, np.pi / 180)["err"] is not None:
            s -= 1
        if s > 2:
            assert setup(1, s - 1, rho, np.pi / 180)["err"] is None
            assert s / float(F32(rho)) < K["MAGIC_RHO"], (rho, s)
    assert setup(1, 12285, 1, np.pi / 180)["apc"] == 1 and setup(1, 6142, 0.5, np.pi / 180)["err"] == "unsupported"


def test_standalone_images_reach_their_cases():
    """Every vote class, prediction class, privatised-copy regime and flush, apc value, per value with nseg below and
    not a multiple of it, and both RS parities are reached by the standalone images; the skipped middle bin is not."""
    cases = standalone_cases()
    tot, regimes, apcs, pers, rs_par, near90, offsets = _coverage(cases)
    assert all(tot[k] > 0 for k in CLASSES + PRED if k != "three_mid_skipped"), tot
    assert tot["three_mid_skipped"] == 0, tot
    assert regimes == {("seg", "single"), ("seg", "atomic"), ("votes", "atomic"), ("par", "atomic")}, regimes
    assert apcs == {1, 2, 4, 8, 16, 32}
    assert {p for p, below, rem in pers if rem} >= {2, 4, 8, 16, 32} and any(below for _, below, _ in pers)
    assert rs_par == {0, 1} and near90 > 0
    for rho in (20, 5, 2, 1, 0.5):
        assert offsets[rho] == set(range(31)), (rho, sorted(set(range(31)) - offsets[rho]))
    na = {setup(c[1].shape[0], c[1].shape[1], c[2], c[3])["na"] for c in cases}
    assert {180, 360, 31, 6, 3, 1} <= na
    # per image: what it was built for
    by = {}
    for name, img, rho, theta, thr in cases:
        o = vote_paths(img, setup(img.shape[0], img.shape[1], rho, theta))
        for k in CLASSES + PRED + ("near90",):
            by.setdefault(name, dict.fromkeys(CLASSES + PRED + ("near90",), 0))[k] += o[k]
    assert all(by["boundary_words"][k] for k in ("two", "three_mid_set", "three_mid_empty", "pixel_coarse", "pixel_fine"))
    assert by["near90"]["off_by_more"] > 0 and by["near90"]["near90"] > 0
    tcfg = setup(64, 96, 2, np.pi / 180)
    assert ties(img_ties(), tcfg, [0]) > 0 and ties(img_ties(), tcfg, [90]) > 0
    assert tables(180, 2, np.pi / 180)[0][90] == F32(0.5) and tables(180, 2, np.pi / 180)[1][90] != 0


def test_peak_images_reach_every_tie_kind():
    """Each of k_hough_peaks' four neighbour comparisons is decided by equality somewhere, and peaks sit in the first
    and last angle row and rho column."""
    tot = dict.fromkeys(PEAK_KINDS, 0)
    for img in img_peaks():
        for rho in (1, 3, 20):
            if setup(img.shape[0], img.shape[1], rho, np.pi / 180)["err"] is None:
                _, acc, _ = cr.hough_lines(img, rho, np.pi / 180, 0)
                for k, v in peak_kinds(acc, 0).items():
                    tot[k] += v
    assert all(tot.values()), tot


# ---- GPU tests ------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def handle():
    from lfd_b200 import _lib
    h = _lib.Handle(8, 8, max_batch=1)
    yield h
    h.close()


def _same(got, ref):
    if ref is None or got is None:
        return ref is None and got is None
    return got.shape == ref.shape and np.array_equal(got.view(np.uint32), ref.view(np.uint32))


def _check_standalone(h, cv2, img, rho, theta, thr, counter=True):
    """lfd_hough_lines against cv2.HoughLines and the oracle: accumulator, line list, n_lines, counter 13."""
    errs = []
    got, acc = h.hough_lines(img, rho, theta, thr, want_accum=True)
    ref_lines, racc, _ = cr.hough_lines(img, rho, theta, thr)
    cvl = cv2.HoughLines(img, rho, theta, thr)
    if not np.array_equal(acc, racc):
        errs.append("accumulator differs at %d cells" % int((acc != racc).sum()))
    if not _same(got, cvl):
        errs.append("lines differ from cv2: %s vs %s" % (None if got is None else got.shape, None if cvl is None else cvl.shape))
    if not _same(got, ref_lines):
        errs.append("lines differ from the oracle")
    if h.last_n_lines != (0 if cvl is None else len(cvl)):
        errs.append("n_lines %d vs %d" % (h.last_n_lines, 0 if cvl is None else len(cvl)))
    o = None
    if counter:
        o = vote_paths(img, setup(img.shape[0], img.shape[1], rho, theta))
        if h.counters()["hough_smem_atomics"] != o["atomics"]:
            errs.append("counter 13: %d vs restated %d" % (h.counters()["hough_smem_atomics"], o["atomics"]))
    return errs, o, acc


@pytest.mark.gpu
@pytest.mark.parametrize("group", ["boundary_words", "ties", "near90", "edges", "tall", "wide", "apc", "nchunks"])
def test_standalone_matches_cv2_and_oracle(handle, cv2mod, group):
    """Accumulator cell for cell, line list bit for bit, n_lines and counter 13 on the images built for each vote path,
    frame edge, apc / per split and privatised-copy regime."""
    seen = dict.fromkeys(CLASSES + PRED, 0)
    for name, img, rho, theta, thr in standalone_cases():
        if not name.startswith(group):
            continue
        errs, o, _ = _check_standalone(handle, cv2mod, img, rho, theta, thr)
        assert not errs, "%s %s rho %s theta %s:\n%s" % (name, img.shape, rho, theta, "\n".join(errs))
        for k in seen:
            seen[k] += o[k]
    print(group, seen)


@pytest.mark.gpu
def test_peak_thresholds_and_plateaus(handle, cv2mod):
    """Thresholds 0, 1, max - 1 and max (no line: None, n_lines 0) on the boundary-word image, and the plateau and
    border images at threshold 0."""
    img = img_boundary_words()
    _, acc, _ = cr.hough_lines(img, 5, np.pi / 180, 1)
    top = int(acc.max())
    for thr in (0, 1, top - 1, top):
        errs, _, _ = _check_standalone(handle, cv2mod, img, 5, np.pi / 180, thr, counter=thr == 0)
        assert not errs, (thr, errs)
    assert handle.last_n_lines == 0
    for img in img_peaks():
        for rho in (1, 3, 20):
            if setup(img.shape[0], img.shape[1], rho, np.pi / 180)["err"] is None:
                errs, _, _ = _check_standalone(handle, cv2mod, img, rho, np.pi / 180, 0)
                assert not errs, (img.shape, rho, errs)


@pytest.mark.gpu
@pytest.mark.parametrize("npk", [0, 1, 2, 1023, 1024, 1025, 2048, 5000])
def test_sort_orders_ties_and_truncates(handle, cv2mod, npk):
    """k_hough_sort on exactly npk isolated peaks with many equal votes (ties ordered by accumulator index): the list
    equals cv2.HoughLines, and max_lines in {1, npk - 1, npk, npk + 1} truncates it and still reports npk."""
    rng = np.random.default_rng(npk)
    votes = rng.integers(1, 5, max(npk, 1))
    img = img_sort(votes)
    thr = int(votes.max()) if npk == 0 else 0
    errs, _, acc = _check_standalone(handle, cv2mod, img, 1, 3.0, thr)
    assert not errs, errs
    assert handle.last_n_lines == npk
    ref = cv2mod.HoughLines(img, 1, 3.0, thr)
    for ml in sorted({1, max(npk - 1, 0), npk, npk + 1}):
        got, _ = handle.hough_lines(img, 1, 3.0, thr, max_lines=ml)
        assert handle.last_n_lines == npk
        k = min(ml, npk)
        assert _same(got, None if k == 0 else ref[:k]), (npk, ml)


@pytest.mark.gpu
def test_shared_memory_and_accumulator_limits(handle, cv2mod):
    """numrho 24 573 (apc 1) is exact; numrho 24 574 is LFD_E_UNSUPPORTED; more than 2e8 cells is LFD_E_ARG; after
    each refusal the same handle is exact again."""
    from lfd_b200 import _lib
    small = img_edges(37, 33)
    img = np.zeros((1, 12285), np.uint8)
    img[0, ::97] = 255
    img[0, -1] = 255
    assert setup(1, 12285, 1, np.pi / 180)["nr"] == 24573
    errs, _, _ = _check_standalone(handle, cv2mod, img, 1, np.pi / 180, 0)
    assert not errs, errs
    for shape, rho, theta, code in (((1, 6142), 0.5, np.pi / 180, _lib.LFD_E_UNSUPPORTED), ((10, 340), 1, 1e-5, _lib.LFD_E_ARG)):
        with pytest.raises(_lib.LfdError) as e:
            handle.hough_lines(np.full(shape, 255, np.uint8), rho, theta, 1)
        assert e.value.code == code
        errs, _, _ = _check_standalone(handle, cv2mod, small, 3, np.pi / 180, 0)
        assert not errs, errs


@pytest.mark.gpu
def test_standalone_handles_keep_their_own_buffers(cv2mod):
    """Two handles of different frame sizes on one device, their calls interleaved across image sizes, rho and theta
    (theta = 3.0: a single angle), are each exact; after one handle is closed the other is exact again."""
    from lfd_b200 import _lib
    a, b = _lib.Handle(8, 8, max_batch=1), _lib.Handle(64, 96, max_batch=1)
    try:
        calls = [(a, img_edges(37, 33), 3, np.pi / 180), (b, img_ties(), 2, np.pi / 180), (a, img_ties(), 1, 3.0),
                 (b, img_edges(37, 33), 1, 3.0), (a, img_edges(120, 200), 1, np.pi / 90), (b, img_ties(), 5, np.pi / 180),
                 (a, img_edges(120, 200), 5, np.pi / 180), (b, img_edges(120, 200), 2, 3.0)]
        for h, img, rho, theta in calls + calls:
            errs, _, _ = _check_standalone(h, cv2mod, img, rho, theta, 0)
            assert not errs, (img.shape, rho, theta, errs)
        a.close()
        for h, img, rho, theta in calls:
            if h is b:
                errs, _, _ = _check_standalone(b, cv2mod, img, rho, theta, 0)
                assert not errs, (img.shape, rho, theta, errs)
    finally:
        a.close()
        b.close()


@pytest.mark.gpu
def test_standalone_handles_on_two_devices(cv2mod):
    """One handle on each of two devices, the same image size on both: every call runs on its own device's buffers."""
    from lfd_b200 import _lib
    handles = []
    try:
        for dev in (0, 1):
            try:
                handles.append(_lib.Handle(8, 8, max_batch=1, device=dev))
            except _lib.LfdError as e:
                if "no such CUDA device" not in str(e):
                    raise
                pytest.skip("fewer than two CUDA devices visible")
        for img, rho, theta in ((img_ties(), 2, np.pi / 180), (img_ties(), 1, 3.0), (img_edges(64, 96), 5, np.pi / 90)):
            for h in handles + handles:
                errs, _, _ = _check_standalone(h, cv2mod, img, rho, theta, 0)
                assert not errs, (h.device, img.shape, rho, theta, errs)
    finally:
        for h in handles:
            h.close()


# ---- the pipeline's Hough, k_check_theta and k_finalize --------------------------------------------------------------
# (H, W, frames, houghMethod values): W % 32 == 12 (handles need W % 4 == 0), and the production frame
BATCHES = [(160, 332, 24, (20, 5, 2, 1)), (1489, 2048, 6, (20,))]


def batch_frames(H, W, n):
    """n frames: empty (zeros, sky only), stars without a line (no rectangle passes), bright trails, faint trails that
    only the dim pass sees, and crossing trails whose line sets disagree."""
    from lfd_b200 import synth
    rng = np.random.default_rng(77)
    L1, L2 = 0.42 * W, 0.36 * W
    frames = []
    for f in range(n):
        kind = f % 6
        trails = []
        if kind in (2, 4, 5):
            a = rng.uniform(0, np.pi)
            trails.append({"p0": (W / 2 - L1 * np.cos(a), H / 2 - L1 * np.sin(a)),
                           "p1": (W / 2 + L1 * np.cos(a), H / 2 + L1 * np.sin(a)), "sigma": 1.5, "peak": 3.0})
        if kind in (3, 4):
            a = rng.uniform(0, np.pi)
            trails.append({"p0": (W / 3 - L2 * np.cos(a), H / 3 - L2 * np.sin(a)),
                           "p1": (W / 3 + L2 * np.cos(a), H / 3 + L2 * np.sin(a)), "sigma": 2.0,
                           "peak": 0.2 if kind == 3 else 3.0})
        img, _ = synth.make_frame(900 + f, n_stars=(0 if kind == 0 else 25 * (W // 332)), trails=trails, h=H, w=W)
        if f in (0, 12):
            img[:] = 0
        frames.append(img)
    return np.stack(frames).astype(np.float32)


def theta_stats(r, p, navg):
    """k_check_theta's four statistics in float64, in the kernel's order: |mean rho1 - mean rho2|, theta spread of
    each set, mean |theta1 - theta2|."""
    n1, n2 = r.n_lines_equ[p], r.n_lines_box[p]
    ro1, ro2, t1, t2 = (np.zeros(navg) for _ in range(4))
    for i in range(navg):
        if i < n1:
            ro1[i] = r.top_equ[p][i][0]
            if i < n2:
                ro2[i], t1[i], t2[i] = r.top_box[p][i][0], r.top_equ[p][i][1], r.top_box[p][i][1]
    s1 = s2 = sd = 0.0
    for i in range(navg):
        s1 += ro1[i]
        s2 += ro2[i]
        sd += abs(t1[i] - t2[i])
    return abs(s1 / navg - s2 / navg), abs(t1.max() - t1.min()), abs(t2.max() - t2.min()), sd / navg


def rejection(stats, dro, thetaTresh, lineSetTresh):
    """0 = accepted, else the 1-based index of the test that rejects."""
    for i, thr in enumerate((dro, thetaTresh, thetaTresh, lineSetTresh)):
        if stats[i] > thr:
            return i + 1
    return 0


def _verdict(r, shape):
    from lfd_b200.processfield import result_from_device
    for p in (0, 1):
        if r.rect_detection[p] >= 0:
            d_, o_ = result_from_device(r, p, shape)
            if d_:
                return (True, p, o_)
    return (False, -1, None)


@pytest.mark.gpu
@pytest.mark.parametrize("H,W,n,rhos", BATCHES)
def test_batch_hough_check_theta_and_finalize(cv2mod, H, W, n, rhos):
    """A 24-frame batch of 160 x 332 frames at houghMethod 20, 5, 2 and 1 (six production-size frames at 20), overlapped and with SERIAL_PASSES, KEEP_TAPS | FULL_LINES: for
    every frame and pass where Hough ran, the accumulators equal the oracle's on that frame's own morph and box taps,
    the line lists equal cv2.HoughLines, top_equ / top_box hold the first nlinesInSet lines (1, 3, 16) with zeros past
    n_lines, counter 13 equals the restated sum, and verdict, pass, rho, theta, status and rejected equal
    oracle.ref_pipeline.  A handle max_lines truncates the lists.  k_check_theta: each statistic as its own threshold
    accepts, nextafter below it rejects; every rejection reason and acceptance occurs."""
    from lfd_b200 import _lib
    frames = batch_frames(H, W, n)
    fl = _lib.KEEP_TAPS | _lib.FULL_LINES
    h = _lib.Handle(H, W, max_batch=n)
    hl = _lib.Handle(H, W, max_batch=n, max_lines=5)
    cache, outcomes = {}, set()
    try:
        def run(handle, pb, pd, flags, nl):
            handle.set_params(dict(pb, nlinesInSet=nl), dict(pd, nlinesInSet=nl))
            handle.submit(frames, flags=flags)
            return handle.wait()

        def check(handle, res, rho, nl, max_lines=None):
            errs, atomics = [], 0
            for f in range(n):
                r = res[f]
                for p in (0, 1):
                    morph, box = handle.stage(f, p, "morph"), handle.stage(f, p, "box")
                    ran = bool(box.any())
                    if r.rect_detection[p] >= 0 and r.rect_detection[p] != int(ran):
                        errs.append("frame %d pass %d: rect_detection %d, box image %s" % (f, p, r.rect_detection[p], ran))
                    if not ran:
                        continue
                    key = (rho, f, p)
                    if key not in cache:
                        ent = {"taps": (morph, box)}
                        for which, src in (("equ", morph), ("box", box)):
                            ent[which] = (cr.hough_lines(src, rho, np.pi / 180, 1)[1], cv2mod.HoughLines(src, rho, np.pi / 180, 1),
                                          vote_paths(src, setup(H, W, rho, np.pi / 180))["atomics"])
                        cache[key] = ent
                    ent = cache[key]
                    if not (np.array_equal(morph, ent["taps"][0]) and np.array_equal(box, ent["taps"][1])):
                        errs.append("frame %d pass %d: taps differ between runs" % (f, p))
                    for which in ("equ", "box"):
                        acc, lines, a13 = ent[which]
                        atomics += a13
                        if not np.array_equal(handle.stage(f, p, "accum_" + which).reshape(acc.shape), acc):
                            errs.append("frame %d pass %d: accum_%s differs" % (f, p, which))
                        if r.rect_detection[p] < 0:
                            continue        # the dim pass of a frame bright decided: k_finalize reports it as not run
                        npk = 0 if lines is None else len(lines)
                        got = handle.stage(f, p, "lines_" + which)
                        k = npk if max_lines is None else min(npk, max_lines)
                        if not _same(got if len(got) else None, lines[:k] if k else None):
                            errs.append("frame %d pass %d: lines_%s differ" % (f, p, which))
                        nrep = r.n_lines_equ[p] if which == "equ" else r.n_lines_box[p]
                        top = np.ctypeslib.as_array(r.top_equ[p] if which == "equ" else r.top_box[p]).astype(np.float32)[:nl]
                        want = np.zeros((nl, 2), np.float32)
                        want[:min(nl, npk)] = lines[:min(nl, npk), 0]
                        if nrep != npk or not np.array_equal(top.view(np.uint32), want.view(np.uint32)):
                            errs.append("frame %d pass %d: top_%s / n_lines differ" % (f, p, which))
            if handle.counters()["hough_smem_atomics"] != atomics:
                errs.append("counter 13: %d vs restated %d" % (handle.counters()["hough_smem_atomics"], atomics))
            return errs

        for rho in rhos:
            pb, pd = dict(rp.DEFAULT_BRIGHT, houghMethod=rho), dict(rp.DEFAULT_DIM, houghMethod=rho)
            taps = [{} for _ in range(n)]
            ref = [rp.process_frame(frames[f].copy(), None, "r", pb, pd, taps=taps[f]) for f in range(n)]
            for flags in (fl, fl | _lib.SERIAL_PASSES):
                for nl in ((1, 3, 16) if rho == 20 and flags == fl else (3,)):
                    res = run(h, pb, pd, flags, nl)
                    errs = check(h, res, rho, nl)
                    assert not errs, "rho %s flags %d nlines %d:\n%s" % (rho, flags, nl, "\n".join(errs[:20]))
                    for f in range(n):
                        r = res[f]
                        assert r.status == 0, (rho, f, r.status)
                        if nl == 3:
                            assert _verdict(r, (H, W)) == tuple(ref[f]), (rho, f, _verdict(r, (H, W)), ref[f])
                        for p, tp, pp in ((0, taps[f]["bright"], pb), (1, taps[f]["dim"], pd)):
                            if r.rect_detection[p] != 1 or not tp or tp.get("lines_equ") is None:
                                continue
                            want = bool(rp.check_theta(tp["lines_equ"], tp["lines_box"], nl, pp["dro"], pp["thetaTresh"],
                                                       pp["lineSetTresh"]))
                            assert r.rejected[p] == int(want), (rho, f, p, nl)
                            outcomes.add(rejection(theta_stats(r, p, nl), pp["dro"], pp["thetaTresh"], pp["lineSetTresh"]))
                        outcomes.add("det%d" % ref[f][1] if ref[f][0] else ("norect" if r.rect_detection[0] == 0 and
                                                                             r.rect_detection[1] == 0 else "rejected"))
        # handle max_lines
        pb, pd = dict(rp.DEFAULT_BRIGHT), dict(rp.DEFAULT_DIM)
        errs = check(hl, run(hl, pb, pd, fl, 3), 20, 3, max_lines=5)
        assert not errs, "max_lines 5:\n" + "\n".join(errs[:20])
        # k_check_theta at exactly each statistic and just below it
        res = run(h, pb, pd, fl, 3)
        stats = {f: theta_stats(res[f], 0, 3) for f in range(n) if res[f].rect_detection[0] == 1}
        big = 1e300
        for i, name in enumerate(("dro", "thetaTresh", "thetaTresh", "lineSetTresh")):
            cand = [f for f, s in stats.items() if (i != 1 or s[1] >= s[2]) and (i != 2 or s[2] > s[1])]
            if not cand and n < 24:
                continue            # the production-size batch is too small to hold every case; the other one does
            assert cand, name
            f = max(cand, key=lambda g: stats[g][i])
            for thr, want in ((stats[f][i], 0), (np.nextafter(stats[f][i], -np.inf), i + 1)):
                p = dict(pb, dro=big, thetaTresh=big, lineSetTresh=big)
                p[name] = float(thr)
                rr = run(h, p, pd, fl, 3)
                assert rejection(stats[f], p["dro"], p["thetaTresh"], p["lineSetTresh"]) == want
                for g, s in stats.items():
                    assert rr[g].rejected[0] == int(rejection(s, p["dro"], p["thetaTresh"], p["lineSetTresh"]) > 0), (name, g)
                outcomes.add(want)
        print("outcomes", sorted(map(str, outcomes)))
        assert n < 24 or {0, 1, 2, 3, 4, "det0", "det1", "norect"} <= outcomes, outcomes
    finally:
        h.close()
        hl.close()
