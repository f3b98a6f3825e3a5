"""The morphology kernels and the Sobel / non-maximum suppression kernels, exactly, on every dispatch path, at their
strip, chunk and tile seams and on the rows and units they skip.

Which kernel runs is a host decision (lfd_b200.cu, run_pass_kernels; lfd_b200/_lib.py, Handle.set_params):
  morphology  k_morph_any for a non-rectangular element or a rectangle whose reach exceeds the tile halo
              (eh//2 + dh//2 > 16 or ew//2 + dw//2 > 11); else k_morph_march<EH, EW, DH, DW> when W % 8 == 0 and the
              shape is one of the MORPH_CASE instantiations; else the k_morph tile kernel;
  NMS         k_nms_march when W % 8 == 0, else the k_canny_nms tile kernel; <true> with LFD_KEEP_TAPS, <false> in
              untapped runs and in lfd_canny.
morph_kernel() / nms_kernel() restate that choice, and the MORPH_CASE list and the strip, chunk and tile constants are
read from the CUDA sources.  Every image is built from those constants and asserts on the CPU what it reaches (ring
phases, skipped units next to processed ones, units that see input only in their halo, pixels on both sides of each
NMS sector boundary), so a change of MARCH_UW, MARCH_R, NMS_R or of the instantiation list cannot quietly retire a
case.  Every comparison is bit-exact against oracle/ref_pipeline.py's pass taps, oracle/cv_restate.py or cv2.Canny.
The morphology kernel's non-zero mask has no tap: it is observed through the Hough accumulator of the equalised
plane and the nnz_equ counter."""
import math
import os
import re

import numpy as np
import pytest

from oracle import cv_restate as cr
from oracle import ref_pipeline as rp

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "lfd_b200", "csrc")


def _read(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _define(src, name):
    return int(re.search(r"#define\s+%s\s+(\d+)" % name, src).group(1))


_MORPH_SRC, _CANNY_SRC = _read("k_morph.cuh"), _read("k_canny.cuh")
MARCH_UW, MARCH_R = _define(_MORPH_SRC, "MARCH_UW"), _define(_MORPH_SRC, "MARCH_R")
MORPH_TW, MORPH_TH = _define(_MORPH_SRC, "MORPH_TW"), _define(_MORPH_SRC, "MORPH_TH")
NMS_R = _define(_CANNY_SRC, "NMS_R")
CANNY_TW, CANNY_TH = _define(_CANNY_SRC, "CANNY_TW"), _define(_CANNY_SRC, "CANNY_TH")
MORPH_CASES = [tuple(int(v) for v in m) for m in
               re.findall(r"^\s*MORPH_CASE\((\d+),\s*(\d+),\s*(\d+),\s*(\d+)\)\s*$", _read("lfd_b200.cu"), re.M)]
STRIP_PX = 4 * MARCH_UW            # useful pixels per strip of both marching kernels
STRIP_MW = STRIP_PX // 32          # mask words per strip

SHAPES = [(1489, 2048),            # production frame: partial last strip, H not a multiple of 64 or 32
          (8, 8),                  # the smallest frame, smaller than a 9- or 15-row element
          (72, 448),               # two whole strips, one 64-row chunk plus 8 rows
          (97, 232),               # the second strip holds one word pair
          (130, 516), (33, 12)]    # W % 8 == 4: the tile kernels
PROD = SHAPES[0]
HALO_SIDES = ("left", "centre", "above", "below", "right")       # the index staggers the probed units


def _ones(h, w):
    return np.ones((h, w), np.uint8)


# (bright dilate, dim erode, dim dilate); the other parameters are the defaults, with addFlux = 0 so that gray == v
PARAM_SETS = {
    "default": ((4, 4), (3, 3), (9, 9)),
    "config4": ((9, 9), (3, 3), (15, 15)),
    "small": ((3, 3), (2, 2), (4, 4)),          # even-sized elements: asymmetric anchors
    "limit": ((33, 23), (3, 3), (31, 21)),      # the tile kernel at its halo limit
    "any": ((3, 24), (3, 3), (3, 24)),          # one column past it: k_morph_any
}


def params(name, shape):
    bd, ee, dd = PARAM_SETS[name]
    lw = 5 if min(shape) >= 64 else 1           # lets a streak pass in the tiny frames too
    pb = dict(rp.DEFAULT_BRIGHT, dilateKernel=_ones(*bd), lwTresh=lw)
    pd = dict(rp.DEFAULT_DIM, erodeKernel=_ones(*ee), dilateKernel=_ones(*dd), addFlux=0.0, lwTresh=lw)
    return pb, pd


# ---- restatement of the kernel choice ------------------------------------------------------------------------------
def morph_kernel(pass_, p, W):
    """('any' | 'march' | 'tile', (eh, ew, dh, dw)) for one pass of a parameter dict."""
    ek = p.get("erodeKernel") if pass_ == 1 else None
    dk = np.asarray(p["dilateKernel"])
    eh, ew = (0, 0) if ek is None else np.asarray(ek).shape
    dh, dw = dk.shape
    shape = (eh, ew, dh, dw)
    all_ones = (ek is None or np.all(np.asarray(ek) != 0)) and np.all(dk != 0)
    if not all_ones or eh // 2 + dh // 2 > 16 or ew // 2 + dw // 2 > 11:
        return "any", shape
    if W % 8 == 0 and shape in MORPH_CASES:
        return "march", shape
    return "tile", shape


def nms_kernel(W):
    return "march" if W % 8 == 0 else "tile"


def reaches(shape):
    """(top, bottom, left, right) reach of erode + dilate with cv2's anchor (k // 2)."""
    eh, ew, dh, dw = shape
    t = eh // 2 + dh // 2
    b = (eh - 1 - eh // 2 if eh else 0) + dh - 1 - dh // 2
    l = ew // 2 + dw // 2
    r = (ew - 1 - ew // 2 if ew else 0) + dw - 1 - dw // 2
    return t, b, l, r


# ---- images --------------------------------------------------------------------------------------------------------
def _seams(n, period, tail):
    out = {0, n - 1}
    for k in range(1, (n + period - 1) // period + 1):
        for v in ((k * period - 1, k * period) if not tail else (k * period - 1, k * period, k * period + period - 1)):
            out.add(v)
    return out


def seam_anchors(H, W, vreach, hreach):
    """(y, x) anchors on every strip, chunk and tile seam and frame edge, each moved by the given reaches."""
    xs = _seams(W, STRIP_PX, True) | _seams(W, MORPH_TW, False) | _seams(W, CANNY_TW, False)
    ys = _seams(H, MARCH_R, False) | _seams(H, NMS_R, False) | _seams(H, MORPH_TH, False) | _seams(H, CANNY_TH, False)
    xs = sorted({x + o for x in xs for o in {0} | {s * v for v in hreach for s in (-1, 1)}} & set(range(W)))
    ys = sorted({y + o for y in ys for o in {0} | {s * v for v in vreach for s in (-1, 1)}} & set(range(H)))
    # x seams on a few chunk seam rows, y seams on the frame's side columns: the frame keeps empty units next to busy ones
    rows = sorted({0, H - 1} | ({MARCH_R - 1, MARCH_R, NMS_R - 1, NMS_R} & set(range(H))))
    cols = [0, W - 1]
    pts = [(rows[i % len(rows)], x) for i, x in enumerate(xs)] + [(y, cols[i % len(cols)]) for i, y in enumerate(ys)]
    return pts + [(0, 0), (0, W - 1), (H - 1, 0), (H - 1, W - 1)]


def put_blocks(img, pts, sizes, rng):
    """k x k blocks of random values 1..255, alternately starting and ending at each anchor, clipped to the frame."""
    H, W = img.shape
    for i, (y, x) in enumerate(pts):
        k = sizes[i % len(sizes)]
        y0, x0 = (y, x) if (i // len(sizes)) % 2 == 0 else (y - k + 1, x - k + 1)
        y0, x0 = max(y0, 0), max(x0, 0)
        img[y0:y0 + k, x0:x0 + k] = rng.integers(1, 256, img[y0:y0 + k, x0:x0 + k].shape)
    return img


def unit_geometry(W):
    """(rows, pixels) of one NMS unit: a k_nms_march strip chunk or a k_canny_nms tile."""
    return (NMS_R, STRIP_PX) if nms_kernel(W) == "march" else (CANNY_TH, CANNY_TW)


def halo_image(H, W, side, shape, rng):
    """Probes whose morphology footprint (element shape `shape`; (0, 0, 1, 1) for the identity) ends exactly on one
    side of an NMS unit: in the mask word left or right of it, or in the rows above or below it.  Every third unit gets
    one, so the unit next to the probe sees it only through its skip window's halo.  'centre' probes sit in the middle
    of every other unit (a checkerboard), so skipped units lie next to processed ones in both orders along both axes."""
    eh, ew, dh, dw = shape
    bh, bw = max(eh, 1), max(ew, 1)                     # an erode-sized block erodes to one pixel at (eh//2, ew//2)
    rh, uw = unit_geometry(W)
    img = np.zeros((H, W), np.float32)
    for c in range((H + rh - 1) // rh):
        for s in range((W + uw - 1) // uw):
            if (c + s + HALO_SIDES.index(side)) % (2 if side == "centre" else 3):
                continue
            y0, y1, x0, x1 = c * rh, min(c * rh + rh, H), s * uw, min(s * uw + uw, W)
            py, px = (y0 + y1) // 2, (x0 + x1) // 2
            if side == "left" and s > 0:
                px = x0 - 1 - dw // 2
            elif side == "right" and x1 < W:
                px = x1 + dw - 1 - dw // 2
            elif side == "above" and c > 0:
                py = y0 - 1 - dh // 2
            elif side == "below" and y1 < H:
                py = y1 + dh - 1 - dh // 2
            elif side != "centre":
                continue
            by, bx = py - bh // 2, px - bw // 2
            if 0 <= by and by + bh <= H and 0 <= bx and bx + bw <= W:
                img[by:by + bh, bx:bx + bw] = rng.integers(1, 256, (bh, bw))
    return img


def streak(img, value=255):
    """A thin line across the frame: after any of the dilations above it is a long thin component whose rectangle
    passes, so Hough runs."""
    H, W = img.shape
    for x in range(W):
        img[min(H // 3 + (x * max(H // 10, 1)) // W, H - 1), x] = value
    return img


def row_pattern(H, lens, gaps):
    """Row flags: non-zero runs of every length in `lens`, each followed by zero runs of every length in `gaps`."""
    flags = np.zeros(H, bool)
    y, cyc = 0, 0
    while y < H:
        for L in lens:
            for g in gaps:
                flags[y:y + L] = True
                y += L + g
        cyc += 1
        flags[y:y + 1] = True       # a one-row run and a longer gap shift the next cycle: the run starts walk
        y += 2 + cyc                # through the ring phases
    return flags


def rows_image(H, W, flags, rng):
    img = np.zeros((H, W), np.float32)
    cols = (np.arange(W) // 5) % 3 != 2                 # 10 px bands of random values, 5 px gaps, in every strip
    img[np.ix_(flags, cols)] = rng.integers(1, 256, (int(flags.sum()), int(cols.sum())))
    return img


def pass_images(H, W, shape, rng):
    """{name: (float32 frame, has_streak)} for one pass whose morphology has element shape `shape`."""
    t, b, l, r = reaches(shape)
    vr, hr = {t, b, t + 1, b + 1}, {l, r, l + 1, r + 1}
    eh, _, dh, _ = shape
    out = {}
    for name, sizes in (("seams_1_3", (1, 3)), ("seams_2_4", (2, 4))):
        out[name] = (streak(put_blocks(np.zeros((H, W), np.float32), seam_anchors(H, W, vr, hr), sizes, rng)), True)
    for side in HALO_SIDES:
        out["halo_" + side] = (halo_image(H, W, side, shape, rng), False)     # a streak would fill their empty units
    rows = rows_image(H, W, row_pattern(H, (1, 2, 3, eh + dh), range(1, dh + 2)), rng)
    out["rows"] = (streak(rows), True)
    out["all255"] = (np.full((H, W), 255, np.float32), False)
    out["const77"] = (np.full((H, W), 77, np.float32), False)
    for k in (1, 4):
        a = np.zeros((H, W), np.float32); a[:k] = 255; a[H - k:] = 255
        out["border_rows_%d" % k] = (streak(a, 128), True)
        a = np.zeros((H, W), np.float32); a[:, :k] = 255; a[:, W - k:] = 255
        out["border_cols_%d" % k] = (streak(a, 128), True)
    # grey values that equalise to 0: 3x3 blocks of 1 and 2 (they survive the erosions), so few next to the bright
    # bottom third that their cumulative count stays below half a LUT step, far from the streak
    low = streak(np.zeros((H, W), np.float32))
    low[2 * H // 3:] = rng.integers(128, 256, (H - 2 * H // 3, W))
    nblk = max((W * (H - 2 * H // 3)) // (600 * 9), 1)
    for i in range(nblk):
        y, x = 2 + 8 * (i // max(W // 8, 1)), 2 + 8 * (i % max(W // 8, 1))
        low[y:y + 3, x:x + 3] = 1 + (i % 2 if nblk > 1 else 0)
    out["low"] = (low, True)
    out["dense"] = (streak(rng.integers(0, 256, (H, W)).astype(np.float32)), True)
    return out


# ---- what the images reach -----------------------------------------------------------------------------------------
def unit_grid(nz, kind):
    """(window_any, core_any, halo kinds) per NMS unit of k_nms_march ('march') or tile of k_canny_nms ('tile'), from
    the non-zero mask of the NMS input.  Halo kinds: 1 left word, 2 right word, 4 rows above, 8 rows below."""
    H, W = nz.shape
    WW = (W + 31) // 32
    words = np.zeros((H, WW * 32), bool)
    words[:, :W] = nz
    words = words.reshape(H, WW, 32).any(axis=2)
    rh, ww = (NMS_R, STRIP_MW) if kind == "march" else (CANNY_TH, CANNY_TW // 32)
    nr, nc = (H + rh - 1) // rh, (WW + ww - 1) // ww
    win, core, halo = np.zeros((nr, nc), bool), np.zeros((nr, nc), bool), np.zeros((nr, nc), int)
    for c in range(nr):
        y0, y1 = c * rh, min(c * rh + rh, H)
        ra, rb = max(y0 - 2, 0), min(y1 + 1, H - 1)
        for s in range(nc):
            w0, w1 = s * ww, min(s * ww + ww, WW)
            wa, wb = max(w0 - 1, 0), min(w0 + ww, WW - 1)
            win[c, s] = words[ra:rb + 1, wa:wb + 1].any()
            core[c, s] = words[y0:y1, w0:w1].any()
            if win[c, s] and not core[c, s]:
                halo[c, s] = (1 * words[y0:y1, wa:w0].any() + 2 * words[y0:y1, w1:wb + 1].any()
                              + 4 * words[ra:y0, wa:wb + 1].any() + 8 * words[y1:rb + 1, wa:wb + 1].any())
    return win, core, halo


def skip_neighbours(win):
    """Which of (skipped left of processed, processed left of skipped, skipped above processed, processed above
    skipped) occur."""
    s = ~win
    return {"h+": bool((s[:, :-1] & win[:, 1:]).any()), "h-": bool((win[:, :-1] & s[:, 1:]).any()),
            "v+": bool((s[:-1] & win[1:]).any()), "v-": bool((win[:-1] & s[1:]).any())}


def check_nms_units(nzs, W, H, what):
    """Over a set of NMS inputs of one frame shape: skipped units next to processed ones in both orders along every axis
    where the geometry allows it, and units that see input only through each side of their halo."""
    kind = nms_kernel(W)
    seen, halo = {}, 0
    for nz in nzs:
        win, _core, h = unit_grid(nz, kind)
        for k, v in skip_neighbours(win).items():
            seen[k] = seen.get(k, False) or v
        for bit in (1, 2, 4, 8):
            if (h == bit).any():
                halo |= bit
    rh, uw = unit_geometry(W)
    want = {a + "-" for a, n, u in (("h", (W + 31) // 32, uw // 32), ("v", H, rh)) if n > u}
    # skipped before processed needs a unit whose core leaves its predecessor's window (the 8-px last strip does not)
    want |= {a + "+" for a, n, u, hw in (("h", (W + 31) // 32, uw // 32, 1), ("v", H, rh, 2))
             if any(min(i * u + 2 * u, n) > min(i * u + u + hw, n) for i in range((n + u - 1) // u - 1))}
    assert want <= {k for k, v in seen.items() if v}, (what, seen)
    want_halo = (3 if W > uw else 0) | (12 if H > rh else 0)
    assert halo & want_halo == want_halo, (what, "halo-only units reached: %d of %d" % (halo, want_halo))


def ring_phases(flags, shape):
    """Ring phases (row - first row of its chunk's march) % lcm(EH, DH) at which non-zero runs start."""
    eh, _, dh, _ = shape
    U = max(eh, 1) * dh // math.gcd(max(eh, 1), dh)
    starts = np.flatnonzero(flags & ~np.concatenate([[False], flags[:-1]]))
    return {int((y - ((y // MARCH_R) * MARCH_R - dh // 2 - eh // 2)) % U) for y in starts}, U


def run_gap_pairs(flags):
    """{(non-zero run length, following zero run length)} of a row pattern (runs cut by the frame end excluded)."""
    out, y, H = set(), 0, len(flags)
    while y < H:
        if flags[y]:
            e = y
            while e < H and flags[e]:
                e += 1
            g = e
            while g < H and not flags[g]:
                g += 1
            if g < H:
                out.add((e - y, g - e))
            y = g
        else:
            y += 1
    return out


def sobel(img):
    """(dx, dy) of cv2.Sobel(ksize=3) with BORDER_REPLICATE, int32."""
    p = np.pad(img.astype(np.int32), 1, mode="edge")
    a = lambda dy, dx: p[1 + dy:1 + dy + img.shape[0], 1 + dx:1 + dx + img.shape[1]]
    dx = (a(-1, 1) + 2 * a(0, 1) + a(1, 1)) - (a(-1, -1) + 2 * a(0, -1) + a(1, -1))
    dy = (a(1, -1) + 2 * a(1, 0) + a(1, 1)) - (a(-1, -1) + 2 * a(-1, 0) + a(-1, 1))
    return dx, dy


def sector_sides(img, low=0):
    """{(boundary, sign of dx, sign of dy, side)} over pixels with magnitude > low lying within one unit of |dy| of the
    22.5 or 67.5 degree sector boundary (OpenCV's integer tests |dy| << 15 vs |dx| * 13573 and + |dx| << 16)."""
    dx, dy = sobel(img)
    ax, ay = np.abs(dx).astype(np.int64), np.abs(dy).astype(np.int64) << 15
    live = (np.abs(dx) + np.abs(dy) > low) & (dx != 0) & (dy != 0)
    out = set()
    for name, t in (("22", ax * 13573), ("67", ax * 13573 + (ax << 16))):
        for side, m in (("below", (ay < t) & (ay > t - (1 << 15))), ("above", (ay >= t) & (ay < t + (1 << 15)))):
            for sx in (-1, 1):
                for sy in (-1, 1):
                    if (live & m & (np.sign(dx) == sx) & (np.sign(dy) == sy)).any():
                        out.add((name, sx, sy, side))
    return out


def sector_image(H, W, rng):
    """Noisy ramps in 16 x 16 patches, their slopes at or near 22.5 and 67.5 degrees in all four quadrants, plus
    plateaus and exact ramps along each direction (equal magnitudes next to each other: the > / >= rules)."""
    img = np.zeros((H, W), np.uint8)
    yy, xx = np.mgrid[0:16, 0:16]
    i = 0
    for py in range(0, H - 15, 16):
        for px in range(0, W - 15, 16):
            kind = i % 6
            if kind < 4:
                ang = (22.5, 67.5)[kind % 2] + rng.uniform(-3, 3) + 90 * rng.integers(0, 4)
                s = rng.uniform(2, 6)
                v = 128 + s * (np.cos(np.radians(ang)) * (xx - 8) + np.sin(np.radians(ang)) * (yy - 8)) + rng.normal(0, 0.7, (16, 16))
            elif kind == 4:
                d = i // 6 % 4
                v = (40 + 6 * (xx, yy, xx + yy, xx - yy + 15)[d]).astype(np.float64)
            else:
                v = np.full((16, 16), 50.0); v[4:12, 4:12] = 50 + 10 * (1 + i // 6 % 5)
            img[py:py + 16, px:px + 16] = np.clip(np.rint(v), 0, 255).astype(np.uint8)
            i += 1
    return img


def nms_images(H, W, rng):
    """uint8 inputs of lfd_canny: seams, row gaps of 1..4 zero rows, sector boundaries / thresholds, dense noise."""
    out = {}
    for name, sizes in (("seams_1_3", (1, 3)), ("seams_2_4", (2, 4))):
        out[name] = put_blocks(np.zeros((H, W), np.uint8), seam_anchors(H, W, {1, 2}, {1, 2}), sizes, rng)
    for side in HALO_SIDES:
        out["halo_" + side] = halo_image(H, W, side, (0, 0, 1, 1), rng).astype(np.uint8)
    out["gaps"] = rows_image(H, W, row_pattern(H, (1, 2), (1, 2, 3, 4)), rng).astype(np.uint8)
    out["sectors"] = sector_image(H, W, rng) if min(H, W) >= 16 else rng.integers(0, 256, (H, W)).astype(np.uint8)
    out["dense"] = rng.integers(1, 256, (H, W)).astype(np.uint8)
    return out


def thresholds(img):
    """(lo, hi): magnitudes lo, lo + 1, hi and hi + 1 all occur at pixels NMS keeps."""
    cls, mag = cr.canny_classes(img, 0, 0)
    vals = set(np.unique(mag[cls != 0]).tolist())
    pairs = sorted(v for v in vals if v + 1 in vals and v > 0)
    if len(pairs) < 2:
        return 10, 100
    return pairs[len(pairs) // 4], pairs[(3 * len(pairs)) // 4]


# ---- oracle --------------------------------------------------------------------------------------------------------
def ref_taps(pass_, img, p):
    taps = {}
    (rp.bright_pass if pass_ == 0 else rp.dim_pass)(img.copy(), taps=taps, **p)
    return taps


# ---- CPU: what the parameter sets and images reach -----------------------------------------------------------------
def test_dispatch_covers_every_instantiation():
    assert MORPH_CASES, "no MORPH_CASE found in lfd_b200.cu"
    reached = {}
    for name in PARAM_SETS:
        for H, W in SHAPES:
            pb, pd = params(name, (H, W))
            for pass_, p in ((0, pb), (1, pd)):
                k, shape = morph_kernel(pass_, p, W)
                reached.setdefault((k, shape), set()).add((name, pass_, W % 8))
    for case in MORPH_CASES:
        passes = {0} if case[0] == 0 else {1}        # the bright pass has no erosion; the dim pass always erodes
        got = {pa for (_n, pa, _w) in reached.get(("march", case), ())}
        assert passes <= got, ("MORPH_CASE%s is not exercised" % (case,), got)
    assert ("default", 0, 4) in reached[("tile", (0, 0, 4, 4))] and ("default", 1, 4) in reached[("tile", (3, 3, 9, 9))]
    assert {("limit", 0, 0), ("limit", 0, 4)} <= reached[("tile", (0, 0, 33, 23))]
    assert {("limit", 1, 0), ("limit", 1, 4)} <= reached[("tile", (3, 3, 31, 21))]
    assert reaches((0, 0, 33, 23))[:3] == (16, 16, 11) and reaches((3, 3, 31, 21))[:3] == (16, 16, 11)
    assert ("any", 0, 0) in reached[("any", (0, 0, 3, 24))] and ("any", 1, 4) in reached[("any", (3, 3, 3, 24))]
    assert ("small", 1, 0) in reached[("tile", (2, 2, 4, 4))]
    t, b, l, r = reaches((2, 2, 4, 4))
    assert (t, l) != (b, r), "even-sized elements must have asymmetric anchors"
    assert {nms_kernel(W) for _H, W in SHAPES} == {"march", "tile"}


def test_row_patterns_cover_every_ring_phase(cv2mod):
    """At the production height, the zero-row image of each marching instantiation has non-zero runs of 1, 2, 3 and
    EH + DH rows followed by zero runs of every length 1 .. DH + 1, starting at every ring phase; under a 3x3 erosion
    the 1- and 2-row runs vanish."""
    rng = np.random.default_rng(0)
    for case in MORPH_CASES:
        eh, _, dh, _ = case
        flags = row_pattern(PROD[0], (1, 2, 3, eh + dh), range(1, dh + 2))
        pairs = run_gap_pairs(flags)
        assert {(L, g) for L in (1, 2, 3, eh + dh) for g in range(1, dh + 2)} <= pairs, case
        phases, U = ring_phases(flags, case)
        assert phases == set(range(U)), (case, sorted(phases), U)
    img = rows_image(PROD[0], 64, row_pattern(PROD[0], (1, 2, 3, 12), range(1, 11)), rng).astype(np.uint8)
    er = cv2mod.erode(img, _ones(3, 3))
    runs = run_gap_pairs(img.any(axis=1))
    assert {1, 2} <= {L for L, _ in runs}
    vanished = img.any(axis=1) & ~er.any(axis=1)
    assert vanished.sum() > 0 and er.any()


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "%dx%d" % s)
def test_nms_images_reach_skips_halos_and_sectors(shape):
    H, W = shape
    rng = np.random.default_rng(H * 7919 + W)
    imgs = nms_images(H, W, rng)
    check_nms_units([v != 0 for k, v in imgs.items() if k not in ("sectors", "dense")], W, H, "lfd_canny %dx%d" % shape)
    win, _, _ = unit_grid(imgs["dense"] != 0, nms_kernel(W))
    assert win.all()
    rows = imgs["gaps"].any(axis=1)
    assert {1, 2, 3} <= {g for _L, g in run_gap_pairs(rows)} or H < 16
    if H * W >= 72 * 232:
        assert len(sector_sides(imgs["sectors"])) == 16, sorted(sector_sides(imgs["sectors"]))
        lo, hi = thresholds(imgs["sectors"])
        assert lo + 1 < hi, (lo, hi)


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "%dx%d" % s)
def test_pass_images_reach_skips_and_zero_lut(shape, cv2mod):
    """The NMS input of the run_pass images (the oracle's morph planes) has skipped units next to processed ones and
    halo-only units; dense noise skips nothing; the low-value image has non-zero grey values that equalise to 0."""
    H, W = shape
    for name in ("default", "limit"):
        pb, pd = params(name, shape)
        for pass_, p in ((0, pb), (1, pd)):
            rng = np.random.default_rng(H * 31 + W + pass_)
            imgs = pass_images(H, W, morph_kernel(pass_, p, W)[1], rng)
            sparse = [k for k in imgs if k.startswith(("seams", "halo")) or k == "rows"]
            morphs = {k: ref_taps(pass_, imgs[k][0], p) for k in sparse + ["low", "dense"]}
            if H >= 64 and name == "default":
                check_nms_units([morphs[k]["morph"] != 0 for k in sparse], W, H, "%s pass %d %dx%d" % (name, pass_, H, W))
            win, _, _ = unit_grid(morphs["dense"]["morph"] != 0, nms_kernel(W))
            assert win.all()
            if H * W >= 72 * 232:
                lt = morphs["low"]
                lut = cr.equalize_lut(np.bincount(lt["gray"].ravel(), minlength=256))
                v = lt["gray"][:H // 3 - 12]
                assert v.any() and not lut[v].any(), (name, pass_)


# ---- GPU -----------------------------------------------------------------------------------------------------------
def _handle(H, W, B=1):
    from lfd_b200 import _lib
    return _lib.Handle(H, W, max_batch=B, max_runs=H * ((W + 1) // 2), max_components=1 << 18)


def _diff(name, got, ref):
    if got.shape != ref.shape:
        return "%s: shape %s vs %s" % (name, got.shape, ref.shape)
    bad = np.argwhere(got != ref)
    if len(bad) == 0:
        return None
    first = [tuple(int(v) for v in b) for b in bad[:4]]
    return "%s: %d differ, first at %s (got, ref)=%s" % (name, len(bad), first, [(got[t].item(), ref[t].item()) for t in first])


@pytest.mark.gpu
@pytest.mark.parametrize("pname", list(PARAM_SETS))
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "%dx%d" % s)
def test_pass_morph_nms_exact(shape, pname, cv2mod):
    """Tapped and untapped run_pass on every pass image: gray, lut, equ, eroded, morph, nms and canny bit-exact, lut[0]
    == 0, and wherever Hough ran, the equalised-plane accumulator and nnz_equ equal those of the oracle's morph plane."""
    from lfd_b200 import _lib
    H, W = shape
    pb, pd = params(pname, shape)
    h = _handle(H, W)
    try:
        h.set_params(pb, pd)
        for pass_, p in ((0, pb), (1, pd)):
            k, eshape = morph_kernel(pass_, p, W)
            rng = np.random.default_rng(H * 1000003 + W * 101 + pass_)
            hough_seen = 0
            for iname, (img, has_streak) in pass_images(H, W, eshape, rng).items():
                if iname == "dense" and shape == PROD and pname not in ("default", "config4"):
                    continue
                tag = "%s/%s pass %d %dx%d (%s)" % (pname, iname, pass_, H, W, k)
                taps = ref_taps(pass_, img, p)
                r = h.run_pass(pass_, img.copy(), flags=_lib.KEEP_TAPS, writeback=False)
                assert not (r.status & _lib.FRAME_OVERFLOW), tag
                errs = []
                for stage in ("gray", "equ", "morph", "canny") + (("eroded",) if pass_ == 1 else ()):
                    errs.append(_diff(stage, h.stage(0, pass_, stage), taps[stage]))
                lut = h.stage(0, pass_, "lut")
                errs.append(_diff("lut", lut, cr.equalize_lut(np.bincount(taps["gray"].ravel(), minlength=256))))
                assert lut[0] == 0, tag
                errs.append(_diff("nms", h.stage(0, pass_, "nms"), cr.canny_classes(taps["morph"], 0, 255)[0]))
                ran = h.counters()["frames_hough"]
                assert ran == (1 if taps["passing"] else 0), (tag, ran, len(taps["passing"]))
                if ran:
                    hough_seen += 1
                    _, acc, _ = cr.hough_lines(taps["morph"], p["houghMethod"], np.pi / 180, 1)
                    errs.append(_diff("accum_equ", h.stage(0, pass_, "accum_equ").reshape(acc.shape), acc))
                    nnz = h.counters()["nnz_equ"]
                    if nnz != np.count_nonzero(taps["morph"]):
                        errs.append("nnz_equ %d vs %d" % (nnz, np.count_nonzero(taps["morph"])))
                errs = [e for e in errs if e]
                assert not errs, tag + ": " + "; ".join(errs)
                # untapped: k_nms_march<false> (or k_canny_nms without its tap)
                r = h.run_pass(pass_, img.copy(), flags=0, writeback=False)
                assert not (r.status & _lib.FRAME_OVERFLOW), tag
                for stage in ("morph", "canny"):
                    e = _diff(stage, h.stage(0, pass_, stage), taps[stage])
                    assert e is None, tag + " untapped: " + e
            if min(H, W) >= 64:
                assert hough_seen >= 1, (pname, pass_, shape, hough_seen)
    finally:
        h.close()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "%dx%d" % s)
def test_canny_standalone_exact(shape, cv2mod):
    """lfd_canny (k_nms_march<false> or k_canny_nms on the packed input mask) against cv2.Canny: low == high, where the
    edge map is the whole candidate mask, and low < high, at thresholds that kept magnitudes hit exactly."""
    H, W = shape
    rng = np.random.default_rng(H * 7919 + W)
    h = _handle(H, W)
    try:
        h.set_params(dict(rp.DEFAULT_BRIGHT), dict(rp.DEFAULT_DIM))
        for iname, img in nms_images(H, W, rng).items():
            lo, hi = thresholds(img)
            for a, b in ((lo, lo), (hi, hi), (0, 0), (lo, hi), (lo + 1, hi + 1), (0, 255)):
                ref = cv2mod.Canny(img, a, b)
                e = _diff("edges", h.canny(img, a, b), ref)
                assert e is None, "%s %dx%d canny(%d, %d) [%s]: %s" % (iname, H, W, a, b, nms_kernel(W), e)
    finally:
        h.close()


@pytest.mark.gpu
@pytest.mark.parametrize("serial", [False, True], ids=["overlapped", "serial"])
def test_batch_taps_per_frame(serial, cv2mod):
    """One KEEP_TAPS batch of 20 different production frames (different LUTs, three without any non-zero pixel): each
    frame's morph and nms taps equal the oracle's on that frame's flipped input, in every pass that ran."""
    from lfd_b200 import _lib
    H, W = PROD
    rng = np.random.default_rng(2024)
    pb, pd = dict(rp.DEFAULT_BRIGHT), dict(rp.DEFAULT_DIM)
    src = pass_images(H, W, (0, 0, 4, 4), rng)
    names = ["seams_1_3", "seams_2_4", "rows", "border_rows_4", "border_cols_4", "low"]
    frames = []
    for i in range(20):
        if i in (0, 9, 19):
            frames.append(np.zeros((H, W), np.float32))
            continue
        f = src[names[i % len(names)]][0].copy()
        f = np.where(f > 0, np.minimum(f * (0.25 + 0.15 * i) + i, 255), 0).astype(np.float32)   # a different LUT each
        frames.append(np.ascontiguousarray(f[::-1] if i % 2 else f))
    frames = np.stack(frames)
    h = _handle(H, W, 20)
    try:
        h.set_params(pb, pd)
        h.submit(frames, [np.zeros((0, 4), np.int32)] * 20, flags=_lib.KEEP_TAPS | (_lib.SERIAL_PASSES if serial else 0))
        res = h.wait()
        dims = 0
        for i in range(20):
            assert not (res[i].status & _lib.FRAME_OVERFLOW), i
            work = np.ascontiguousarray(frames[i][::-1]).copy()
            tb, td = {}, {}
            rp.bright_pass(work, taps=tb, **pb)
            rp.dim_pass(work, taps=td, **pd)
            for pass_, taps in ((0, tb), (1, td)):
                if res[i].rect_detection[pass_] < 0:
                    assert pass_ == 1, i
                    continue
                dims += pass_
                for e in (_diff("morph", h.stage(i, pass_, "morph"), taps["morph"]),
                          _diff("nms", h.stage(i, pass_, "nms"), cr.canny_classes(taps["morph"], 0, 255)[0])):
                    assert e is None, "frame %d pass %d: %s" % (i, pass_, e)
        assert dims >= 10
    finally:
        h.close()
