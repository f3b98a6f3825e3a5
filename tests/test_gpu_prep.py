"""The input stage, exactly: k_star_mask, k_prep<MODE, BE> on every path, k_prep_generic, k_lut and k_blot
(lfd_b200/csrc/k_prep.cuh, lfd_b200.cu).

k_prep<0, BE> (lfd_submit) gives every warp a TMA ring of 2 KB chunks, one chunk being 512 pixels of a row; a row
whose byte length is not a multiple of 2 KB ends in a partial chunk of nf4 < 128 float4.  A warp walks the chunks
pc, pc + stride, ... of a frame (row step dy, chunk step dj, with a wrap of pj when stride % cpr != 0), and its CTA
walks the frames blockIdx.y, blockIdx.y + 16, ..., carrying the mbarrier phase across them.  Words (four output
bytes) with a byte >= 2 go to a per-warp staging list of PR_STG words per plane, drained when it holds more than
PR_STG - 32 * PR_Q words before a chunk is staged; hist4_fix then corrects bin 1 of the dp4a byte sums.  The mask
words of a chunk are fetched one chunk ahead, skipped with one vote and spread to the lanes by __shfl_sync.
launch() and walk() restate the grid of run_pipeline and the chunk walk; their constants are read from the CUDA
sources, so changing one fails a test instead of quietly retiring a case.  The number of resident CTAs per SM cannot
be observed from Python, so every coverage test holds for each occupancy the shared memory allows (1..4) at 148
SMs; test_device_grid_is_covered repeats the assertions with the SM count of the device the GPU tests run on.

The conversions are compared bit for bit with NumPy's clips (processfield.py:342, 453-454; under NumPy 2 a Python
float scalar is cast to float32 first, which test_numpy_scalar_semantics pins) followed by cv2.convertScaleAbs and
oracle/cv_restate.py, the histograms with np.bincount and the LUT with cv2.equalizeHist.  The parameter grid holds
minFlux <= 0 (the denormal threshold of the folded dim compare), negative addFlux (negative sums, the exact redo) and
float32 neighbours of every rounding edge.

k_prep_generic's mode-0 branches (mask, flip, both planes) are unreachable from the library: only lfd_run_pass asks
for the clipped plane, and it runs mode 1 or 2.  They remain the reference of the k_prep micro-benchmark
(profiles/lab/prep_lab.cu) and are not tested here."""
import functools
import os
import re

import numpy as np
import pytest

from oracle import cv_restate as cr
from oracle import ref_pipeline as rp

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "lfd_b200", "csrc")
F32 = np.float32
SMS = 148                           # B200 SMs: the coverage tests' grid
SMEM_PER_SM, SMEM_RESERVED = 228 * 1024, 1024


def _read(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


_PREP, _CU = _read("k_prep.cuh"), _read("lfd_b200.cu")


def _constants():
    c = {}
    for k in ("PR_WARPS", "PR_S", "PR_Q", "PR_CF4", "PR_CB", "PR_STG", "PR_SMEM"):
        expr = re.search(r"^#define\s+%s\s+([^/\n]+)" % k, _PREP, re.M).group(1)
        c[k] = int(eval(expr, {"__builtins__": {}}, dict(c)))
    drains = re.findall(r"if \(nst([01]) > ([^)]+)\) drain_big\(stg\1, nst\1,", _PREP)
    assert [p for p, _ in drains] == ["0", "1"] and drains[0][1] == drains[1][1], drains
    c["DRAIN"] = int(eval(drains[0][1], {"__builtins__": {}}, dict(c)))
    gy = re.search(r"const int gy = n < (\d+) \? n : (\d+);", _CU).groups()
    assert gy[0] == gy[1], gy
    c["GY"] = int(gy[0])
    for pat in (r"int rb = h->prep_grid\[mode\] / gy; if \(rb < 1\) rb = 1;",
                r"const int chunks = d\.H \* \(\(d\.W \* 4 \+ PR_CB - 1\) / PR_CB\);",
                r"if \(rb > \(chunks \+ PR_WARPS - 1\) / PR_WARPS\) rb = \(chunks \+ PR_WARPS - 1\) / PR_WARPS;",
                r"h->prep_grid\[m\] = prop\.multiProcessorCount \* \(per_sm\[m\] > 0 \? per_sm\[m\] : 1\);",
                r"const int stride = gridDim\.x \* PR_WARPS;",
                r"pc \+= stride; py \+= dy; pj \+= dj; if \(pj >= cpr\) \{ pj -= cpr; py\+\+; \}"):
        assert re.search(pat, _CU + _PREP), pat
    return c


C = _constants()
PR_WARPS, PR_Q, PR_CF4, PR_CB, PR_STG, DRAIN, GY = (C[k] for k in ("PR_WARPS", "PR_Q", "PR_CF4", "PR_CB", "PR_STG",
                                                                   "DRAIN", "GY"))
MASK_WORDS = PR_CB // 4 // 32       # star-mask words per chunk
OCCS = range(1, SMEM_PER_SM // (C["PR_SMEM"] + SMEM_RESERVED) + 1)
MAX_RECTS = 8192                    # lfd_config.max_star_rects default


# ---- restatement of the launch and the chunk walk -------------------------------------------------------------------
def launch(H, W, n, occ, sms=SMS):
    """(cpr, total chunks per frame, gy, rb, stride) of run_pipeline's k_prep launch."""
    cpr = -(-4 * W // PR_CB)
    total = H * cpr
    gy = min(n, GY)
    rb = min(max(sms * occ // gy, 1), -(-total // PR_WARPS))
    return cpr, total, gy, rb, rb * PR_WARPS


def nf4_of(W, j):
    return min(PR_CF4, (4 * W - j * PR_CB) >> 4)


def walk(H, W, n, occ, sms=SMS):
    """Yields (frame, warp, chunks, wraps): the flat chunk indices one warp converts in one frame, in order, and how
    often its pj wrapped.  The kernel's incremental (py, pj) is restated and checked against pc."""
    cpr, total, gy, rb, stride = launch(H, W, n, occ, sms)
    dy, dj = divmod(stride, cpr)
    for by in range(gy):
        for f in range(by, n, gy):
            for w in range(rb * PR_WARPS):
                pc = w
                py, pj = divmod(pc, cpr)
                seq, wraps = [], 0
                while pc < total:
                    assert py * cpr + pj == pc
                    seq.append(pc)
                    pc += stride
                    py += dy
                    pj += dj
                    if pj >= cpr:
                        pj -= cpr
                        py += 1
                        wraps += 1
                yield f, w, seq, wraps


def chunk_big(g, cpr):
    """(H, cpr): words with a byte >= 2 in each chunk of an output plane."""
    H, W = g.shape
    words = (g.reshape(H, W // 4, 4) >= 2).any(2)
    pad = np.zeros((H, cpr * PR_CF4), bool)
    pad[:, :W // 4] = words
    return pad.reshape(H, cpr, PR_CF4).sum(2)


def chunk_mask_words(mflip, cpr):
    """(H, cpr, MASK_WORDS) bool: which star-mask words of each chunk are non-zero (flipped orientation)."""
    H, W = mflip.shape
    pad = np.zeros((H, cpr * PR_CB // 4), bool)
    pad[:, :W] = mflip
    return pad.reshape(H, cpr, MASK_WORDS, 32).any(3)


def staging(counts0, counts1):
    """The two staging lists of one warp over its chunks, plane 0 staged before plane 1 as in the kernel.  Per plane:
    mid-frame drains, the largest count staged, and whether a chunk of PR_CF4 big words found exactly DRAIN + 1 words
    staged; and whether such a chunk on plane 0 also staged plane-1 words into an empty list (a plane-0 list that
    ran past PR_STG would have lost its last word there)."""
    nst, drains, top, edge = [0, 0], [0, 0], [0, 0], [False, False]
    shared = False
    for c in zip(counts0, counts1):
        hit0 = False
        for p in (0, 1):
            if c[p] == 0:
                continue
            if nst[p] > DRAIN:
                e = nst[p] == DRAIN + 1 and c[p] == PR_CF4
                edge[p] |= e
                hit0 |= e and p == 0
                drains[p] += 1
                nst[p] = 0
            shared |= hit0 and p == 1 and nst[1] == 0
            nst[p] += c[p]
            assert nst[p] <= PR_STG
            top[p] = max(top[p], nst[p])
    return drains, top, edge, shared


@functools.lru_cache(maxsize=None)
def chunk_counts(name):
    """Per frame, (bright, dim) big words of every chunk (flat chunk index) under the case's first parameters."""
    case = CASES[name]
    frames, rects = batch(name)
    cpr = -(-4 * case["W"] // PR_CB)
    out = []
    for f in range(case["n"]):
        _, g0, g1 = ref_planes(frames[f], rects[f], *case["params"][0])
        out.append((chunk_big(g0, cpr).ravel(), chunk_big(g1, cpr).ravel()))
    return out


def coverage(case, occ, sms=SMS):
    """What one case's batch reaches at one occupancy."""
    H, W, n = case["H"], case["W"], case["n"]
    cpr, total, gy, rb, stride = launch(H, W, n, occ, sms)
    out = {"drain": {0: set(), 1: set()}, "full": set(), "edge": set(), "partial_big": set(), "wraps": 0, "shared": False,
           "dj": stride % cpr, "odd_walked": False, "nf4": {nf4_of(W, j) for j in range(cpr)}}
    big = chunk_counts(case["name"])
    for f in range(n):
        for p in (0, 1):
            b = big[f][p].reshape(H, cpr)
            for j in range(cpr):
                if nf4_of(W, j) < PR_CF4 and b[:, j].any():
                    out["partial_big"].add(nf4_of(W, j))
    for f, w, seq, wraps in walk(H, W, n, occ, sms):
        out["wraps"] += wraps
        if len(seq) % 2 and f + gy < n:
            out["odd_walked"] = True
        drains, top, edge, shared = staging(big[f][0][seq], big[f][1][seq])
        out["shared"] |= shared
        for p in (0, 1):
            if drains[p]:
                out["drain"][p].add(f)
            if top[p] == PR_STG:
                out["full"].add(p)
            if edge[p]:
                out["edge"].add(p)
    return out


def mask_reach(case):
    """{(k, partial)} of chunks whose only non-zero mask word is k, and whether such a chunk blots column W - 1."""
    H, W, n = case["H"], case["W"], case["n"]
    frames, rects = batch(case["name"])
    cpr = -(-4 * W // PR_CB)
    ks, last = set(), False
    kl = ((W - 1) % 512) // 32
    for f in range(n):
        m = rect_mask(H, W, rects[f])[::-1]
        cw = chunk_mask_words(m, cpr)
        one = cw.sum(2) == 1
        for y, j in zip(*np.nonzero(one)):
            k = int(np.argmax(cw[y, j]))
            ks.add((k, nf4_of(W, j) < PR_CF4))
            if j == cpr - 1 and k == kl and m[y, W - 1]:
                last = True
    return ks, last


# ---- references -----------------------------------------------------------------------------------------------------
def rect_mask(H, W, rects):
    """Union of the rectangles (r0, r1, c0, c1), half-open, clamped to the frame (k_star_mask / k_blot)."""
    m = np.zeros((H, W), bool)
    for r0, r1, c0, c1 in np.asarray(rects, np.int64).reshape(-1, 4):
        r0, r1, c0, c1 = max(r0, 0), min(r1, H), max(c0, 0), min(c1, W)
        if r0 < r1 and c0 < c1:
            m[r0:r1, c0:c1] = True
    return m


def dim_clip(t, minFlux, addFlux):
    """processfield.py:453-454 in place, with the scalars cast to float32 once, as the library does."""
    with np.errstate(all="ignore"):
        t[t < F32(minFlux)] = 0
        t[t > 0] += F32(addFlux)
    return t


def ref_planes(frame, rects, minFlux, addFlux):
    """(flipped mask, bright gray, dim gray) of one whole-frame run."""
    H, W = frame.shape
    m = rect_mask(H, W, rects)
    t = frame.copy()
    t[m] = 0
    t = np.ascontiguousarray(t[::-1])
    with np.errstate(all="ignore"):
        t[t < 0] = 0
        g0 = cr.convert_scale_abs(t)
        g1 = cr.convert_scale_abs(dim_clip(t, minFlux, addFlux))
    return m[::-1], g0, g1


# ---- images ---------------------------------------------------------------------------------------------------------
BYTES = np.array([0, 1, 2, 3, 127, 128, 129, 254, 255], F32)
COUNTS = (0, 0, 1, 2, 31, 64, 65, 127, 128, 128, 128)


def special_values(minFlux, addFlux):
    vals = [0.0, -0.0, 0.5, 1.5, 2.5, 127.5, 128.5, 254.5, 255.5, 256.0, 1000.0, 2.0 ** 31, -2.0 ** 31, 2147483520.0,
            2.0 ** 31 + 256, 3e9, -3e9, np.inf, -np.inf, 1e-30, -1e-30, 8388608.0, 8388607.5, 16777216.0, -0.25, -0.3]
    v = np.array(vals, F32)
    bits = np.array([0x7fc00000, 0xffc00000, 0x7f800001, 0x7fc12345, 0xff812345, 0xffffffff, 0x00000001, 0x007fffff,
                     0x80000001, 0x807fffff, 0x5700003c, 0x4b0000ff, 0x4b8000aa, 0x4affffff, 0x4b000100], np.uint32)
    centres = []
    with np.errstate(all="ignore"):
        for c in (F32(minFlux), F32(255.5) - F32(addFlux), F32(0.5) - F32(addFlux)):
            if np.isfinite(c):
                centres += [c, -c]
    nb = []
    for c in centres:
        lo = hi = F32(c)
        nb.append(lo)
        for _ in range(3):
            lo, hi = np.nextafter(lo, F32(-np.inf)), np.nextafter(hi, F32(np.inf))
            nb += [lo, hi]
    return np.concatenate([v, bits.view(F32), np.array(nb, F32)])


def sky(rng, shape):
    return rng.normal(0, 0.03, shape).astype(F32)


def put_specials(rng, img, minFlux, addFlux):
    """Every special value three times at random places, and once in the last column."""
    H, W = img.shape
    sp = special_values(minFlux, addFlux)
    ys, xs = rng.integers(0, H, 3 * len(sp)), rng.integers(0, W, 3 * len(sp))
    img[ys, xs] = np.tile(sp, 3)
    img[rng.integers(0, H, len(sp)), W - 1] = sp
    return img


def big_words(rng, k, vals):
    """(k, 4) pixel values from `vals`, each row holding at least one of vals[must:] (a byte >= 2 in the plane)."""
    vals, must = vals
    v = rng.choice(vals, (k, 4))
    need = ~np.isin(v, vals[must:]).any(1)
    v[need, rng.integers(0, 4, need.sum())] = rng.choice(vals[must:], need.sum())
    return v


# (big-word values with the index from which a value is big, small values): every byte of BYTES in the bright plane
# (and, at minFlux 0.02 / addFlux 0.5, in the dim plane too); dim-only big words at addFlux 1.5
FILLS = {"bright": ((BYTES, 2), np.array([0.0, 1.0, 0.4, -2.0], F32)),
         "both": ((BYTES, 2), np.array([0.0, 0.4, -2.0, 0.01], F32)),
         "dim": ((np.array([0.0, 0.01, 0.3, 0.8, 1.2], F32), 2), np.array([0.0, 0.01, -3.0, 1e-30], F32))}


def fill_counts(rng, H, W, kind):
    """An output-orientation image whose chunks hold a random number of big words (COUNTS, capped at nf4)."""
    bigv, small = FILLS[kind]
    cpr = -(-4 * W // PR_CB)
    img = rng.choice(small, (H, W)).astype(F32)
    w4 = img.reshape(H, W // 4, 4)
    for y in range(H):
        for j in range(cpr):
            nf4 = nf4_of(W, j)
            k = min(int(rng.choice(COUNTS)), nf4)
            if k:
                pos = j * PR_CF4 + rng.permutation(nf4)[:k]
                w4[y, pos] = big_words(rng, k, bigv)
    return img


def all_bright(rng, H, W):
    """Every pixel converts to a byte >= 2 in both planes at the default parameters."""
    return rng.choice(BYTES[2:], (H, W)).astype(F32)


def single_pixel_rects(H, W, f, nsp):
    """Part f of nsp of one-pixel rectangles at every column: row x % H, and columns of one row at least 512 apart,
    so a chunk holds one blotted pixel."""
    xs = np.arange(W)
    xs = xs[(xs // H) % nsp == f]
    return np.stack([xs % H, xs % H + 1, xs, xs + 1], 1).astype(np.int32)


def edge_rects(H, W, rng):
    """Rectangles clipped by every frame edge, empty after clipping, overlapping, and with edges on word and chunk
    boundaries."""
    r = [(-5, 3, 10, 20), (H - 3, H + 7, 1, 9), (1, 4, -4, 3), (2, 5, W - 2, W + 9), (-2, 2, -2, 2),
         (H - 1, H + 1, W - 1, W + 1),                                                     # clipped
         (-9, -1, 0, 5), (-9, 0, 0, 5), (H, H + 4, 0, 5), (3, 3, 0, 5), (6, 2, 0, 5), (0, 5, W, W + 5),
         (0, 5, -7, 0), (0, 5, 9, 4), (-100, -50, -100, -50), (H + 1, H + 9, W + 1, W + 9)]  # empty
    r += [(2, 6, 3, 9), (4, 8, 5, 12), (3, 4, 0, W)]                                         # overlapping
    for i, c in enumerate((31, 32, 33, 63, 64, 480, 511, 512, 513, 544, 1023, 1024, 1536, 2047, W - 33, W - 32)):
        for k, (a, b) in enumerate(((c, c + 1), (c - 1, c + 1), (c, c + 33), (c - 32, c))):
            y = (3 * i + k) % H
            r.append((y, y + 1 + k % 2, a, b))
    r += [tuple(int(v) for v in (y, y + rng.integers(1, 9), x, x + rng.integers(1, 40)))
          for y, x in zip(rng.integers(-5, H + 5, 40), rng.integers(-30, W + 30, 40))]
    return np.array(r, np.int32)


def brighten_under(frame, rects):
    """Blotted pixels must be visible: pixels under a rectangle that are zero-ish get a bright value."""
    H, W = frame.shape
    m = rect_mask(H, W, rects)
    with np.errstate(invalid="ignore"):
        dark = m & ~(np.abs(frame) >= 2)
    frame[dark] = 77.0
    return frame


PARAMS_DEFAULT = (0.02, 0.5)
PARAM_GRID = [(0.02, 0.5), (0.0, -0.25), (-0.0, -0.3), (-1.0, -0.5), (1e-45, -0.75), (3.0, -1.5), (300.0, 0.1),
              (np.inf, 254.5), (np.nan, 255.5), (0.02, 1e10), (0.0, 0.0), (-1.0, -0.0), (1e-45, 0.5), (-0.0, 1.5),
              (0.0, 254.5), (0.02, -0.3)]

CASES = {c["name"]: c for c in [
    dict(name="prod1", H=1489, W=2048, n=1, params=[PARAMS_DEFAULT, (-1.0, -0.75)]),
    dict(name="prod24", H=1489, W=2048, n=24, params=[PARAMS_DEFAULT]),
    dict(name="drain_bright", H=600, W=2048, n=17, params=[(200.0, 0.5)]),
    dict(name="drain_dim", H=600, W=2048, n=17, params=[(0.02, 1.5)]),
    dict(name="w516", H=67, W=516, n=40, params=PARAM_GRID),
    dict(name="w1020", H=33, W=1020, n=40, params=[PARAMS_DEFAULT, (-1.0, -0.5), (0.0, 254.5)]),
    dict(name="w1500", H=40, W=1500, n=40, params=[PARAMS_DEFAULT]),
    dict(name="w2100", H=130, W=2100, n=40, params=[PARAMS_DEFAULT, (-0.0, 1.5)]),
    dict(name="tiny", H=8, W=8, n=3, params=PARAM_GRID),
    dict(name="small", H=33, W=12, n=5, params=[PARAMS_DEFAULT, (0.0, -0.25)]),
]}


@functools.lru_cache(maxsize=None)
def batch(name):
    """(frames (n, H, W) float32 un-flipped, rectangles per frame) of one case."""
    case = CASES[name]
    H, W, n = case["H"], case["W"], case["n"]
    rng = np.random.default_rng(sum(map(ord, name)))
    frames = np.empty((n, H, W), F32)
    rects = []
    nsp = -(-512 // H)
    no_rects = {0, n // 2, n - 1} if n >= 5 else {0}
    for f in range(n):
        if name == "prod1":
            img = fill_counts(rng, H, W, "both")[::-1] + sky(rng, (H, W))
            rc = np.concatenate([single_pixel_rects(H, W, 0, 1), edge_rects(H, W, rng)])
        elif name == "prod24":
            if f in (0, 16):
                img = all_bright(rng, H, W)
            elif f in (1, 17):
                img = fill_counts(rng, H, W, "both")[::-1].copy()
            else:
                img = sky(rng, (H, W))
                img[rng.random((H, W)) < 0.002] += 9.0
            if f == 2:
                rc = single_pixel_rects(H, W, 0, 1)
            elif f == 4:                                            # exactly max_star_rects
                y, x = rng.integers(-3, H, MAX_RECTS), rng.integers(-3, W, MAX_RECTS)
                rc = np.stack([y, y + rng.integers(1, 7, MAX_RECTS), x, x + rng.integers(1, 7, MAX_RECTS)], 1)
            else:
                rc = edge_rects(H, W, rng)
        elif name.startswith("drain_"):
            img = fill_counts(rng, H, W, name[6:])
            if name == "drain_bright":                              # at minFlux 200 only 254 / 255 reach the dim plane
                img[img >= 200] = 129.0
                ys, xs = np.nonzero(rng.random((H, -(-W // 512))) < 0.3)
                img[ys, np.minimum(xs * 512 + rng.integers(0, 512, len(xs)), W - 1)] = 255.0
            img = img[::-1].copy()
            rc = edge_rects(H, W, rng)
        elif name in ("tiny", "small"):
            img = sky(rng, (H, W))
            sel = rng.random((H, W)) < 0.3
            img[sel] = rng.choice(BYTES, sel.sum())
            rc = np.array([(f, f + 2, f, f + 3), (-1, 1, W - 2, W + 3), (H - 1, H + 2, -1, 2)] if f % 2 else
                          [(0, H, 4, 5), (3, 2, 0, W)], np.int32)
        else:
            img = fill_counts(rng, H, W, "both")[::-1] + sky(rng, (H, W))
            rc = single_pixel_rects(H, W, f % nsp, nsp) if f < nsp * 2 else edge_rects(H, W, rng)
        if name not in ("drain_bright", "drain_dim") and not (name == "prod24" and f in (0, 16)):
            put_specials(rng, img, *case["params"][f % len(case["params"])])
        rc = np.asarray(rc, np.int32).reshape(-1, 4) if f not in no_rects or name == "prod1" else np.zeros((0, 4), np.int32)
        frames[f] = brighten_under(img, rc)
        rects.append(rc)
    return frames, rects


# ---- CPU: restatement, images and oracle semantics ------------------------------------------------------------------
def test_constants_read_from_sources():
    assert (PR_WARPS, PR_Q, PR_CF4, PR_CB, PR_STG, DRAIN, GY) == (8, 4, 128, 2048, 256, 128, 16)
    assert MASK_WORDS == 16 and list(OCCS) == [1, 2, 3, 4]
    assert PR_STG - DRAIN == PR_CF4             # one chunk stages at most PR_CF4 words: the list never overflows


def test_walk_visits_every_chunk_once():
    for case in CASES.values():
        H, W, n = case["H"], case["W"], case["n"]
        for occ in OCCS:
            cpr, total, gy, rb, stride = launch(H, W, n, occ)
            seen = np.zeros((n, total), np.int64)
            for f, w, seq, _ in walk(H, W, n, occ):
                seen[f, seq] += 1
            assert (seen == 1).all(), (case["name"], occ)


def test_numpy_scalar_semantics():
    """The oracle's clips compare and add in float32 (NumPy 2 casts a Python float scalar to the array's dtype), like
    the library's single (float) cast; if NumPy changes this, the GPU comparisons below would fail obscurely."""
    a = np.array([0.02, 0.1, 0.25], F32)
    assert not (a < 0.02)[0] and np.array_equal(a < 0.02, a < F32(0.02))
    assert float(F32(0.02)) < 0.02              # a float64 comparison would zero this pixel
    b = a.copy()
    b[b > 0] += 0.3
    assert b.dtype == F32 and np.array_equal(b.view(np.uint32), (a + F32(0.3)).view(np.uint32))
    for mf, af in PARAM_GRID:
        t = np.array([F32(mf) if np.isfinite(mf) else 1.0, 0.7], F32)
        u = t.copy()
        with np.errstate(all="ignore"):
            t[t < mf] = 0
            t[t > 0] += af
        assert np.array_equal(t.view(np.uint32), dim_clip(u, mf, af).view(np.uint32)), (mf, af)


@pytest.mark.parametrize("occ", list(OCCS))
def test_batches_reach_every_walk_case(occ):
    assert_walk_cases(occ, SMS)


def assert_walk_cases(occ, sms):
    cov = {name: coverage(CASES[name], occ, sms) for name in CASES}
    # mid-frame drains on both planes, in frame 0 and in a frame a CTA reaches by walking (f >= 16)
    for p in (0, 1):
        d = cov["prod24"]["drain"][p]
        assert 0 in d and any(f >= GY for f in d), (p, d)
    # exactly PR_STG words staged without a drain (128 + 128)
    assert cov["prod24"]["full"] == {0, 1}
    # a chunk of PR_CF4 big words after exactly DRAIN + 1 staged words, on each plane; on plane 0 in a chunk that
    # stages plane-1 words into an empty list, while plane 1 stays below the drain threshold
    assert 0 in cov["drain_bright"]["edge"] and cov["drain_bright"]["shared"], cov["drain_bright"]
    assert not cov["drain_bright"]["drain"][1], cov["drain_bright"]
    assert 1 in cov["drain_dim"]["edge"] and not cov["drain_dim"]["drain"][0], cov["drain_dim"]
    # partial chunks holding big words
    assert 1 in cov["w516"]["partial_big"] and 127 in cov["w1020"]["partial_big"]
    assert cov["w1500"]["nf4"] == {128, 119} and 119 in cov["w1500"]["partial_big"]
    # dj != 0 and pj wraps; an odd chunk count in a frame before the CTA walks on
    assert cov["w2100"]["dj"] != 0 and cov["w2100"]["wraps"] > 0
    assert cov["w2100"]["odd_walked"] and 2100 * 4 % PR_CB != 0


def test_batches_reach_every_mask_word():
    ks, last = mask_reach(CASES["w1020"])
    assert {k for k, part in ks if part} == set(range(MASK_WORDS)) and last
    for name in ("prod1", "w516", "w2100"):
        ks, _ = mask_reach(CASES[name])
        assert {k for k, part in ks if not part} == set(range(MASK_WORDS)), name
    assert mask_reach(CASES["w516"])[1]


def test_batches_hold_their_edge_cases():
    _, rects = batch("prod24")
    assert [len(r) for r in rects].count(0) == 3 and len(rects[0]) == len(rects[12]) == len(rects[23]) == 0
    assert len(rects[4]) == MAX_RECTS
    frames, _ = batch("prod24")
    g = ref_planes(frames[0], rects[0], *PARAMS_DEFAULT)
    assert (g[1] >= 2).all() and (g[2] >= 2).all()
    words = g[1].reshape(-1, 4)
    assert all(np.isin(BYTES.astype(np.uint8)[2:], g[1]))
    assert ((words == 2).any(1) & (words == 255).any(1)).any()
    frames, rects = batch("w516")
    sp = frames.view(np.uint32)
    for b in (0x80000000, 0xffc00000, 0x00000001, 0x80000001, 0x7fc12345):
        assert (sp == b).any(), hex(b)


# ---- LUT histograms --------------------------------------------------------------------------------------------------
LUT_H, LUT_W = 64, 128
LUT_N = LUT_H * LUT_W


def lut_kinds(D, s):
    """Cumulative sums s (over total - h[i0] = D) whose float32 product rounds differently from the exact product
    (kind a), and from 255 * s / D in float32 (kind b)."""
    s = np.asarray(s, np.int64)
    sc = F32(255.0) / F32(D)
    p32 = s.astype(F32) * sc
    a = np.rint(p32) != np.rint(s.astype(np.float64) * np.float64(sc))
    b = np.rint(p32) != np.rint((F32(255.0) * s.astype(F32)) / F32(D))
    return a, b


@functools.lru_cache(maxsize=None)
def lut_histograms():
    """(name, histogram) pairs of LUT_N pixels."""
    out = []

    def add(name, i0, svals):
        """Histogram with h[i0] = LUT_N - D whose bins after i0 reach the cumulative sums svals (increasing, < D),
        the rest of D in bin 255."""
        svals = np.asarray(svals, np.int64)
        h = np.zeros(256, np.int64)
        h[i0 + 1:i0 + 1 + len(svals)] = np.diff(np.concatenate([[0], svals]))
        out.append((name, h))
        return h

    for i0, D, step, n in ((0, 510, 1, 254), (2, 510, 1, 247), (0, 1020, 1, 254), (5, 1020, 3, 249)):
        s = (np.arange(n) + 1) * step + (255 if i0 == 2 else 0)
        h = add("tie%d_%d" % (D, i0), i0, s)
        h[i0] = LUT_N - D
        h[255] += D - s[-1]
    found = []
    for D in range(2, LUT_N):
        a, b = lut_kinds(D, np.arange(1, D))
        if a.any() or b.any():
            found.append((int(a.sum()), int(b.sum()), D, np.nonzero(a | b)[0] + 1))
    picks = sorted(found, key=lambda t: (-t[0], t[2]))[:6] + sorted(found, key=lambda t: (-t[1], t[2]))[:6]
    for k, (_, _, D, s) in enumerate(picks):
        i0 = (0, 3, 17)[k % 3]
        s = s[:250 - i0]
        h = add("search%d" % D, i0, s)
        h[i0] = LUT_N - D
        h[255] += D - s[-1]
    for v in (0, 7, 255):
        h = np.zeros(256, np.int64)
        h[v] = LUT_N
        out.append(("const%d" % v, h))
    for a, na, b in ((0, LUT_N - 5, 200), (3, 1, 9), (254, LUT_N // 2, 255)):
        h = np.zeros(256, np.int64)
        h[a], h[b] = na, LUT_N - na
        out.append(("two%d_%d" % (a, b), h))
    for name, h in out:
        assert h.sum() == LUT_N and (h >= 0).all(), name
    return out


def test_lut_histograms_reach_ties_and_rounding_differences():
    ka = kb = ties = 0
    i0s, h255 = set(), 0
    for name, h in lut_histograms():
        i0 = int(np.nonzero(h)[0][0])
        i0s.add(i0)
        h255 += h[255] > 0 and i0 < 255
        D = LUT_N - h[i0]
        if D == 0:
            continue
        s = np.cumsum(h[i0 + 1:])
        a, b = lut_kinds(D, s)
        ka, kb = ka + a.sum(), kb + b.sum()
        prod = s.astype(F32) * (F32(255.0) / F32(D))
        ties += int((prod - np.floor(prod) == 0.5).sum())
    assert ka >= 36 and kb >= 36 and ties >= 36, (ka, kb, ties)
    assert {0, 3, 7, 17, 255} <= i0s and h255 >= 10


# ---- GPU -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_device_grid_is_covered():
    """The coverage above assumes SMS SMs; the device the GPU tests run on must reach the same cases with its own
    SM count, at every occupancy the shared memory allows."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    for occ in OCCS:
        assert_walk_cases(occ, sms)


def _lib():
    from lfd_b200 import _lib as L
    return L


def params(mf, af):
    return dict(rp.DEFAULT_BRIGHT), dict(rp.DEFAULT_DIM, minFlux=mf, addFlux=af)


def check_whole(h, cv2, frames, rects, mf, af, tag):
    for f in range(len(frames)):
        m, g0, g1 = ref_planes(frames[f], rects[f], mf, af)
        assert np.array_equal(h.stage(f, 0, "mask"), np.where(m, 255, 0).astype(np.uint8)), (tag, f)
        for p, g in ((0, g0), (1, g1)):
            t = frames[f].copy()
            t[m[::-1]] = 0
            t = np.ascontiguousarray(t[::-1])
            with np.errstate(all="ignore"):
                t[t < 0] = 0
            if p:
                dim_clip(t, mf, af)
            assert np.array_equal(cv2.convertScaleAbs(t), g), (tag, f, p)
            got = h.stage(f, p, "gray")
            if not np.array_equal(got, g):
                bad = np.argwhere(got != g)[:5]
                raise AssertionError((tag, f, p, [(tuple(b), got[tuple(b)], g[tuple(b)], t[tuple(b)]) for b in bad]))
            hist = np.bincount(g.ravel(), minlength=256)
            assert np.array_equal(h.stage(f, p, "hist").astype(np.int64), hist), (tag, f, p)
            assert np.array_equal(h.stage(f, p, "lut"), cr.equalize_lut(hist)), (tag, f, p)
            assert np.array_equal(h.stage(f, p, "equ"), cv2.equalizeHist(g)), (tag, f, p)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_whole_frame_prep_matches_numpy_and_cv2(cv2mod, name):
    """k_star_mask and k_prep<0, false> under every parameter pair of the case, then k_prep<0, true> on the same
    batch as big-endian float32: identical planes, and the input tap equals the native frames."""
    L = _lib()
    case = CASES[name]
    frames, rects = batch(name)
    h = L.Handle(case["H"], case["W"], max_batch=case["n"])
    try:
        for k, (mf, af) in enumerate(case["params"]):
            h.set_params(*params(mf, af))
            h.submit(frames, rects, flags=L.KEEP_TAPS)
            h.wait()
            check_whole(h, cv2mod, frames, rects, mf, af, (name, mf, af))
            if k == 0:
                h.submit(np.ascontiguousarray(frames.byteswap()), rects, flags=L.KEEP_TAPS | L.INPUT_BIGENDIAN)
                h.wait()
                check_whole(h, cv2mod, frames, rects, mf, af, (name, mf, af, "BE"))
                for f in range(case["n"]):
                    assert np.array_equal(h.stage(f, 0, "input").view(np.uint32), frames[f].view(np.uint32)), f
    finally:
        h.close()


STANDALONE = [("w1020", 0), ("tiny", 0), ("small", 1), ("w2100", 0), ("prod1", 0)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,frame", STANDALONE)
def test_standalone_passes_match_numpy(name, frame):
    """run_pass: k_prep<1|2, false> without write-back, k_prep_generic with it; the dim pass on unclipped input."""
    L = _lib()
    case = CASES[name]
    img = batch(name)[0][frame]
    grid = PARAM_GRID if case["H"] * case["W"] < 1 << 16 else [PARAMS_DEFAULT, (-1.0, -0.75), (-0.0, 1.5)]
    h = L.Handle(case["H"], case["W"], max_batch=1)
    try:
        for mf, af in grid:
            h.set_params(*params(mf, af))
            for pass_ in (0, 1):
                ref = img.copy()
                if pass_ == 0:
                    with np.errstate(all="ignore"):
                        ref[ref < 0] = 0
                else:
                    dim_clip(ref, mf, af)
                with np.errstate(all="ignore"):
                    g = cr.convert_scale_abs(ref)
                hist = np.bincount(g.ravel(), minlength=256)
                for wb in (False, True):
                    work = img.copy()
                    h.run_pass(pass_, work, flags=L.KEEP_TAPS, writeback=wb)
                    tag = (name, mf, af, pass_, wb)
                    assert np.array_equal(h.stage(0, pass_, "gray"), g), tag
                    assert np.array_equal(h.stage(0, pass_, "hist").astype(np.int64), hist), tag
                    assert np.array_equal(h.stage(0, pass_, "lut"), cr.equalize_lut(hist)), tag
                    expect = ref if wb else img
                    assert np.array_equal(work.view(np.uint32), expect.view(np.uint32)), tag
    finally:
        h.close()


@pytest.mark.gpu
def test_lut_ties_and_rounding(cv2mod):
    """k_lut on histograms of integer-valued frames: .5 ties, float32 products that round differently from the exact
    one, i0 > 0, constant and two-valued frames, h[255] > 0."""
    L = _lib()
    hs = lut_histograms()
    rng = np.random.default_rng(5)
    frames = np.stack([rng.permutation(np.repeat(np.arange(256), h)).reshape(LUT_H, LUT_W).astype(F32) for _, h in hs])
    h = L.Handle(LUT_H, LUT_W, max_batch=len(hs))
    try:
        h.set_params(*params(*PARAMS_DEFAULT))
        h.submit(frames, None, flags=L.KEEP_TAPS)
        h.wait()
        for f, (name, hist) in enumerate(hs):
            got = h.stage(f, 0, "hist").astype(np.int64)
            assert np.array_equal(got, hist), name
            assert np.array_equal(h.stage(f, 0, "lut"), cr.equalize_lut(hist)), name
            g = h.stage(f, 0, "gray")
            assert np.array_equal(h.stage(f, 0, "equ"), cv2mod.equalizeHist(g)), name
            _, _, g1 = ref_planes(frames[f], [], *PARAMS_DEFAULT)
            h1 = np.bincount(g1.ravel(), minlength=256)
            assert np.array_equal(h.stage(f, 1, "lut"), cr.equalize_lut(h1)), name
    finally:
        h.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["w516", "prod1", "small"])
def test_blot_matches_numpy(name):
    L = _lib()
    case = CASES[name]
    H, W = case["H"], case["W"]
    frames, rects = batch(name)
    rc = np.concatenate([edge_rects(H, W, np.random.default_rng(1))] + [r for r in rects if len(r)])
    h = L.Handle(H, W, max_batch=1)
    try:
        for f in range(min(case["n"], 2)):
            img = frames[f].copy()
            ref = img.copy()
            ref[rect_mask(H, W, rc)] = 0
            h.blot(img, rc)
            assert np.array_equal(img.view(np.uint32), ref.view(np.uint32)), (name, f)
        img = frames[0].copy()
        h.blot(img, np.zeros((0, 4), np.int32))
        assert np.array_equal(img.view(np.uint32), frames[0].view(np.uint32))
    finally:
        h.close()


@pytest.mark.gpu
def test_argument_errors_launch_nothing():
    """max_star_rects + 1 rectangles in a frame, rect_offsets[0] != 0 and lfd_run_pass with LFD_INPUT_BIGENDIAN are
    refused with nothing launched; the next call is exact."""
    import ctypes
    L = _lib()
    H, W, n = 33, 1020, 3
    frames, rects = batch("w1020")
    frames, rects = frames[:n].copy(), rects[:n]
    cap = max(len(r) for r in rects)
    h = L.Handle(H, W, max_batch=n, max_star_rects=cap)
    try:
        h.set_params(*params(*PARAMS_DEFAULT))

        def code(fn, *a, **k):
            l0 = h.kernel_launches()
            with pytest.raises(L.LfdError) as e:
                fn(*a, **k)
            assert h.kernel_launches() == l0
            return e.value.code

        def exact(rc):
            h.submit(frames, rc, flags=L.KEEP_TAPS)
            h.wait()
            for f in range(n):
                m, g0, g1 = ref_planes(frames[f], rc[f], *PARAMS_DEFAULT)
                assert np.array_equal(h.stage(f, 0, "mask"), np.where(m, 255, 0).astype(np.uint8)), f
                assert np.array_equal(h.stage(f, 0, "gray"), g0) and np.array_equal(h.stage(f, 1, "gray"), g1), f

        full = [edge_rects(H, W, np.random.default_rng(f))[:cap] for f in range(n)]
        assert all(len(r) == cap for r in full)
        exact(full)
        over = list(full)
        over[1] = np.concatenate([full[1], full[1][:1]])
        assert code(h.submit, frames, over) == L.LFD_E_CAPACITY
        exact(rects)
        flat, offs, _, _ = L.Handle._rects_arrays(full)
        offs = offs + 1
        assert code(lambda: h._ck(h._L.lfd_submit(h.h, frames.ctypes.data_as(ctypes.c_void_p), n,
                                                   flat.ctypes.data_as(ctypes.c_void_p),
                                                   offs.ctypes.data_as(ctypes.c_void_p), 0))) == L.LFD_E_ARG
        exact(full)
        img = np.ascontiguousarray(frames[0][::-1])
        for wb in (False, True):
            work = img.copy()
            assert code(h.run_pass, 0, work, flags=L.INPUT_BIGENDIAN, writeback=wb) == L.LFD_E_ARG
            assert np.array_equal(work.view(np.uint32), img.view(np.uint32))
        h.run_pass(1, img.copy(), writeback=False)
        with np.errstate(all="ignore"):
            g1 = cr.convert_scale_abs(dim_clip(img.copy(), *PARAMS_DEFAULT))
        assert np.array_equal(h.stage(0, 1, "gray"), g1)
        exact(rects)
    finally:
        h.close()
