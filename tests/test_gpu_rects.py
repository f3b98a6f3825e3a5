"""Every contour's rectangle, exactly, on every path of k_rects_warp, and the boxes k_fill_boxes draws from them.

The oracle (oracle/cv_restate.py::rects_and_box) works on the same point sets as the device and starts the calipers at
the same hull vertex, so each device rectangle must be bit-identical to the oracle's one of the same (kind, key); the
multiset comparison of test_gpu_stages.py needs a tolerance only because cv2's hull start vertex follows its trace.

k_rects_warp picks one of these paths per contour (constants of lfd_b200/csrc/k_rects.cuh):
  thread    at most RECT_T_ROWS rows and a thread stack that never exceeds RECT_T_PTS: one thread per contour;
  overflow  at most RECT_T_ROWS rows, but the thread stack would overflow: the warp path, partial chains merged in
            place in shared memory (device counter rects_thread_overflow);
  compact   more rows: per-lane partial chains in global scratch, compacted into shared memory when both chain sums
            are at most RECT_TALL_PTS;
  inplace   the same, chains merged in place in global scratch (the mirrored B regions);
and, orthogonal to compact / inplace, a hull of more than RECT_SMALL_PTS vertices is gathered and walked in global
scratch ("big").  rect_path() restates that choice from a contour's row extremes, so each image below asserts the paths
it was built for: a later change of a constant cannot quietly retire one of these tests."""
import os
import re

import numpy as np
import pytest

from oracle import cv_restate as cr
from oracle import ref_pipeline as rp

HERE = os.path.dirname(os.path.abspath(__file__))
K_RECTS = os.path.join(os.path.dirname(HERE), "lfd_b200", "csrc", "k_rects.cuh")


def _constants():
    with open(K_RECTS) as f:
        src = f.read()
    return {k: int(re.search(r"#define\s+%s\s+(\d+)" % k, src).group(1))
            for k in ("RECT_T_ROWS", "RECT_T_PTS", "RECT_SMALL_PTS", "RECT_TALL_PTS")}


K = _constants()


# ---- restatement of k_rects_warp's path choice ---------------------------------------------------------------------
def _push(st, p, lo):
    """Chain::push: pop while the stack holds at least `lo` entries and the turn is not strictly left."""
    while len(st) >= lo:
        (x2, y2), (x1, y1) = st[-2], st[-1]
        if (x1 - x2) * (p[1] - y2) - (y1 - y2) * (p[0] - x2) > 0:
            break
        st.pop()
    st.append(p)


def _rows(pts):
    """(y0, rows) with rows[r] = (rowmin, rowmax) of the point set, None for an empty row."""
    ys, xs = pts[:, 1], pts[:, 0]
    y0 = int(ys.min())
    hh = int(ys.max()) - y0 + 1
    rmin = np.full(hh, 1 << 30)
    rmax = np.full(hh, -1)
    np.minimum.at(rmin, ys - y0, xs)
    np.maximum.at(rmax, ys - y0, xs)
    return y0, [(int(a), int(b)) if a <= b else None for a, b in zip(rmin, rmax)]


def _thread_overflows(rows):
    """rect_thread_path: the stack check (k + 2 > RECT_T_PTS before each non-empty row) over the ascending and the
    descending chain."""
    st = []
    for r, ab in enumerate(rows):
        if ab is None:
            continue
        if len(st) + 2 > K["RECT_T_PTS"]:
            return True
        _push(st, (ab[0], r), 2)
        if ab[1] != ab[0]:
            _push(st, (ab[1], r), 2)
    n = len(st)
    if n > 1:
        first = True
        for r in range(len(rows) - 1, -1, -1):
            ab = rows[r]
            if ab is None:
                continue
            if len(st) + 2 > K["RECT_T_PTS"]:
                return True
            if first:
                first = False
            else:
                _push(st, (ab[1], r), n + 1)
            if ab[0] != ab[1]:
                _push(st, (ab[0], r), n + 1)
    return False


def _partial_chain_sums(rows):
    """rect_warp_path level 1: each lane's ascending (A) and descending (B) chain over its slice of c = ceil(hh / 32)
    rows; returns (sum of A lengths, sum of B lengths, lanes with an empty slice)."""
    hh = len(rows)
    c = (hh + 31) // 32
    sa = sb = empty = 0
    for lane in range(32):
        r0 = min(lane * c, hh)
        r1 = min(r0 + c, hh)
        empty += r0 == hh
        a, b = [], []
        for r in range(r0, r1):
            if rows[r] is not None:
                _push(a, (rows[r][0], r), 2)
                if rows[r][1] != rows[r][0]:
                    _push(a, (rows[r][1], r), 2)
        for r in range(r1 - 1, r0 - 1, -1):
            if rows[r] is not None:
                _push(b, (rows[r][1], r), 2)
                if rows[r][1] != rows[r][0]:
                    _push(b, (rows[r][0], r), 2)
        sa += len(a)
        sb += len(b)
    return sa, sb, empty


def rect_path(pts):
    """k_rects_warp's path for a contour's point set: dict(path, big, hh, n, empty_lanes)."""
    _, rows = _rows(pts)
    hh = len(rows)
    n = len(cr.hull(pts))
    out = {"hh": hh, "n": n, "big": False, "empty_lanes": 0}
    if hh <= K["RECT_T_ROWS"]:
        out["path"] = "overflow" if _thread_overflows(rows) else "thread"
    else:
        sa, sb, out["empty_lanes"] = _partial_chain_sums(rows)
        out["path"] = "compact" if sa <= K["RECT_TALL_PTS"] and sb <= K["RECT_TALL_PTS"] else "inplace"
        out["big"] = n > K["RECT_SMALL_PTS"]
    return out


# ---- images: each is built for some of those paths ----------------------------------------------------------------
# 2x2 patches whose Canny(0, 255) edge map holds a one-pixel and a two-pixel component (hulls of n = 1 and n = 2)
ONE_PIXEL = np.array([[255, 200], [200, 128]], np.uint8)
TWO_PIXELS = np.array([[128, 200], [60, 255]], np.uint8)


def _pack(H, W, shapes, gap=6):
    """Draw (w, h, draw(img, x, y)) shapes left to right in shelves; shapes that do not fit are left out."""
    img = np.zeros((H, W), np.uint8)
    x = y = gap
    shelf = 0
    for w, h, draw in shapes:
        if x + w + gap > W:
            x, y, shelf = gap, y + shelf + gap, 0
        if y + h + gap > H:
            continue
        draw(img, x, y)
        x += w + gap
        shelf = max(shelf, h)
    return img


def _img_thread(cv2, H, W):
    """Contours of at most RECT_T_ROWS rows: one- and two-pixel components, one-row runs, vertical and diagonal lines
    (collinear hulls), L-shapes, discs up to r = 31, outlines exactly 64 and 65 rows tall, one-pixel holes."""
    def patch(p):
        def d(img, x, y):
            img[y:y + 2, x:x + 2] = p
        return (2, 2, d)

    def fill(w, h):
        def d(img, x, y):
            img[y:y + h, x:x + w] = 255
        return (w, h, d)

    def disc(r):
        return (2 * r + 1, 2 * r + 1, lambda img, x, y: cv2.circle(img, (x + r, y + r), r, 255, -1))

    def line(dx, dy, t):
        return (dx + 1, dy + 1, lambda img, x, y: cv2.line(img, (x, y), (x + dx, y + dy), 255, t))

    def ell(img, x, y):
        img[y:y + 30, x:x + 3] = 255
        img[y + 27:y + 30, x:x + 30] = 255

    shapes = [patch(ONE_PIXEL), patch(TWO_PIXELS), fill(1, 1), fill(2, 1), fill(40, 1), fill(1, 2), fill(1, 60),
              line(40, 40, 1), line(40, 13, 1), line(9, 50, 2), (30, 30, ell), fill(3, 63), fill(3, 64), fill(5, 63),
              fill(7, 64), line(20, 61, 3)]
    shapes += [disc(r) for r in (1, 2, 3, 5, 8, 13, 21, 26, 31)]
    return _pack(H, W, shapes)


def _img_overflow(cv2, H, W):
    """Flat filled ellipses of at most RECT_T_ROWS rows whose hulls overflow the thread stack (outer and hole)."""
    img = np.zeros((H, W), np.uint8)
    a = min(700, W // 2 - 20)
    cv2.ellipse(img, (W // 2, 40), (a, 30), 0, 0, 360, 255, -1)
    if H > 200:
        cv2.ellipse(img, (W // 2, 130), (a * 3 // 4, 26), 3, 0, 360, 255, -1)
    return img


def _img_compact(cv2, H, W):
    """Contours of more rows than RECT_T_ROWS: full-height bars and lines that touch rows 0 and H - 1, long lines at
    several angles, and bars whose outlines are 32k and 32k + 1 rows tall (lanes with empty slices)."""
    img = np.zeros((H, W), np.uint8)
    img[:, 8:11] = 255                                            # full height, vertical
    dx = min(H, W) // 3
    cv2.line(img, (20, 0), (20 + dx, H - 1), 255, 3)             # full height, tilted
    x = 40 + dx
    for n in (64, 95, 96, 127, 128, 255, 256):                 # outlines of n + 1 rows
        if n + 4 < H and x + 12 < W:
            img[2:2 + n, x:x + 3] = 255
            x += 12
    angles = (88, 75, 60, 45, 30, 10)                             # long lines at several angles, one band each
    band = (W - x) // len(angles)
    for i, ang in enumerate(angles):
        c, s = np.cos(np.radians(ang)), np.sin(np.radians(ang))
        L = min((H - 10) / s, (band - 12) / c)
        cv2.line(img, (x, 5), (x + int(L * c), 5 + int(L * s)), 255, 1 + i % 2 * 2)
        x += band
    return img


def _img_inplace(cv2, H, W):
    """Tall contours whose per-lane partial chains exceed RECT_TALL_PTS: 32 discs of r = 55 joined by a 21 px spine,
    one disc per lane slice.  At 4096 x 4096 the spine is the straight side of a half disc of r = 1950, whose round side
    gives the outer and the hole contour more than RECT_SMALL_PTS hull vertices as well."""
    img = np.zeros((H, W), np.uint8)
    if W >= 4096:
        cv2.circle(img, (2100, H // 2), 1950, 255, -1)
        img[:, 2100:] = 0
        for i in range(32):
            cv2.circle(img, (2100, H // 2 - 1950 + 60 + 122 * i), 55, 255, -1)
    else:
        xc = W // 2
        for i in range(32):
            cv2.circle(img, (xc, 64 + 124 * i), 55, 255, -1)
        img[64:64 + 124 * 31, xc - 10:xc + 11] = 255
    return img


def _img_inplace_cut(cv2, H, W):
    """The bead column of _img_inplace leaning by 10 px per bead and cut flat through its last bead: the leftmost pixel
    of the contour's last row is then its only support in the column's direction, so a merge that loses the second
    vertex of the descending chain changes the rectangle."""
    img = np.zeros((H, W), np.uint8)
    centres = [(W - 92 - 10 * i, 64 + 124 * i) for i in range(32)]
    for x, y in centres:
        cv2.circle(img, (x, y), 55, 255, -1)
    cv2.line(img, centres[0], centres[-1], 255, 21)
    img[centres[-1][1] + 20:] = 0
    return img


def _img_big(cv2, H, W):
    """A filled disc whose outer and hole contours have more than RECT_SMALL_PTS hull vertices (compacted chains)."""
    img = np.zeros((H, W), np.uint8)
    r = min(H, W) // 2 - 48
    cv2.circle(img, (W // 2, H // 2), r, 255, -1)
    return img


def _img_edges(cv2, H, W):
    """Shapes cut by column 0, column W - 1, row 0 and row H - 1 and in each corner, tilted so that their boxPoints lie
    outside the frame, and thin lines that leave the frame at a slant."""
    img = np.zeros((H, W), np.uint8)
    s = max(6, min(H, W) // 8)
    centres = [(0, H // 2), (W - 1, H // 3), (W // 3, 0), (2 * W // 3, H - 1),
               (0, 0), (W - 1, 0), (0, H - 1), (W - 1, H - 1), (W // 2, H // 2)]
    for i, (cx, cy) in enumerate(centres):
        box = cv2.boxPoints(((float(cx), float(cy)), (float(3 * s), float(s)), 17.0 + 23 * i))
        cv2.fillPoly(img, [np.int32(np.round(box))], 255)
    cv2.line(img, (W // 4, H // 5), (-W // 8, H // 2), 255, 1)
    cv2.line(img, (3 * W // 4, 4 * H // 5), (W + W // 8, H // 3), 255, 2)
    cv2.line(img, (W // 6, H - H // 6), (W // 3, H + H // 4), 255, 1)
    return img


# (H, W) -> {image: paths it must cover}
SIZES = {
    (1489, 2048): {"thread": {"thread", "compact"}, "overflow": {"overflow"}, "compact": {"compact"},
                   "big": {"compact+big"}, "edges": {"thread", "compact"}},
    (97, 332): {"thread": {"thread", "compact"}, "overflow": {"overflow"}, "compact": {"compact"},
                "edges": {"thread"}},
    (4096, 512): {"compact": {"compact"}, "inplace": {"inplace"}, "inplace_cut": {"inplace"},
                  "edges": {"thread", "compact"}},
    (4096, 4096): {"overflow": {"overflow"}, "big": {"compact+big"}, "inplace": {"inplace+big"},
                   "edges": {"compact"}},
}
BUILDERS = {"thread": _img_thread, "overflow": _img_overflow, "compact": _img_compact, "inplace": _img_inplace,
            "inplace_cut": _img_inplace_cut, "big": _img_big, "edges": _img_edges}


def _contours(edges):
    """{(kind, key): (points, rect_path)} over the oracle's contour sets; kind 0 = outer, 1 = hole."""
    return {(int(k == "hole"), key): (pts, rect_path(pts)) for k, key, pts in cr.contour_point_sets(edges)}


def _tag(p):
    return p["path"] + ("+big" if p["big"] else "")


def _path_counts(contours):
    out = {}
    for _, p in contours.values():
        out[_tag(p)] = out.get(_tag(p), 0) + 1
    return out


def _check_coverage(cv2, H, W, name, contours):
    """The paths (and edges) the image was built for, restated on the CPU."""
    counts = _path_counts(contours)
    missing = SIZES[(H, W)][name] - set(counts)
    assert not missing, "%s at %dx%d no longer reaches %s (paths %s)" % (name, H, W, sorted(missing), counts)
    paths = [p for _, p in contours.values()]
    if name == "thread":
        assert {1, 2} <= {p["n"] for p in paths}
        assert any(p["hh"] == K["RECT_T_ROWS"] and p["path"] == "thread" for p in paths)
        assert any(p["hh"] == K["RECT_T_ROWS"] + 1 and p["path"] == "compact" for p in paths)
        assert any(kind == 1 and p["hh"] == 3 for (kind, _), (_, p) in contours.items())
    if name == "compact":
        tall = [p for p in paths if p["path"] == "compact"]
        assert any(p["hh"] == H for p in tall)
        assert any(p["empty_lanes"] for p in tall)
        if H > 512:
            assert {65, 96, 97, 128, 129} <= {p["hh"] for p in tall}
    if name == "edges":
        boxes = np.array([cr.box_points(cr.min_area_rect(cr.hull(pts))) for pts, _ in contours.values()])
        assert (boxes[..., 0] < 0).any() and (boxes[..., 0] >= W).any()
        assert (boxes[..., 1] < 0).any() and (boxes[..., 1] >= H).any()
    return counts


def _images(cv2, H, W):
    return {name: BUILDERS[name](cv2, H, W) for name in SIZES[(H, W)]}


@pytest.mark.parametrize("H,W", list(SIZES))
def test_images_cover_their_paths(cv2mod, H, W):
    """CPU only: every image reaches the k_rects_warp paths it was built for (restated from the source's constants)."""
    for name, img in _images(cv2mod, H, W).items():
        counts = _check_coverage(cv2mod, H, W, name, _contours(cv2mod.Canny(img, 0, 255)))
        print("%dx%d %s: %s" % (H, W, name, counts))


# ---- device against oracle ----------------------------------------------------------------------------------------
def _bits(*v):
    return tuple(np.array(v, np.float32).view(np.uint32).tolist())


def _handle(H, W, **cfg):
    from lfd_b200 import _lib
    h = _lib.Handle(H, W, max_batch=1, **cfg)
    h.set_params(dict(rp.DEFAULT_BRIGHT), dict(rp.DEFAULT_DIM))
    # lfd_get_stage reads frame slots of the last run: one pass makes slot 0 readable
    h.run_pass(0, np.zeros((H, W), np.float32), writeback=False)
    return h


def _check_rects(rects, box_img, edges, minLen, lwTresh, external=None):
    """A frame's RECTS and BOX taps against the oracle on the same edge map, contour by contour.  `external`: the kind-0
    keys RETR_EXTERNAL retrieves (None: RETR_LIST, every contour).  Returns (errors, contours, detection)."""
    contours = _contours(edges)
    ref_rects, ref_pass, _ = cr.rects_and_box(edges, minLen, lwTresh)
    ref = {(int(k == "hole"), key): r for k, key, r in ref_rects}
    want = set(ref) if external is None else {(0, key) for key in external}
    errs = []
    if len(rects) != len(ref):
        errs.append("%d rects, the oracle has %d contours" % (len(rects), len(ref)))
    seen = set()
    for o in rects:
        kind, key = int(o["kind"]), int(o["key"])
        if kind == 2 and external is not None:          # not retrieved: counted by the caller
            continue
        if (kind, key) in seen or (kind, key) not in want:
            errs.append("rect (%d, %d): %s" % (kind, key, "duplicate" if (kind, key) in seen else "not expected"))
            continue
        seen.add((kind, key))
        (cx, cy), (w, hh), ang = r = ref[(kind, key)]
        length, width = (w, hh) if w > hh else (hh, w)
        passed = length > minLen and width > minLen and length / width > lwTresh
        diff = []
        if _bits(o["cx"], o["cy"], o["w"], o["h"], o["angle"]) != _bits(cx, cy, w, hh, ang):
            diff.append("rect %s vs %s" % ((float(o["cx"]), float(o["cy"]), float(o["w"]), float(o["h"]), float(o["angle"])),
                                           (cx, cy, w, hh, ang)))
        if bool(o["passed"]) != passed:
            diff.append("passed %d vs %d" % (o["passed"], passed))
        elif passed and not np.array_equal(o["box"], cr.box_points(r).astype(np.int32).ravel()):
            diff.append("box %s vs %s" % (o["box"].tolist(), cr.box_points(r).astype(np.int32).ravel().tolist()))
        if diff:
            p = contours[(kind, key)][1]
            errs.append("(%d, %d) rows %d hull %d path %s: %s" % (kind, key, p["hh"], p["n"], _tag(p), "; ".join(diff)))
    if seen != want:
        errs.append("%d contours without a rect" % len(want - seen))
    ref_box = np.zeros(edges.shape, np.uint8)
    passing = [box for kind, key, _, box in ref_pass if (int(kind == "hole"), key) in want]
    for box in passing:
        cr.fill_poly(ref_box, box, 255)
    if not np.array_equal(box_img, ref_box):
        errs.append("box image differs at %d pixels" % int((box_img != ref_box).sum()))
    return errs, contours, bool(passing)


def _fit(h, cv2, img, mode=1, minLen=0.0, lwTresh=0.5):
    """lfd_fit_min_area_rect on img against cv2.Canny and the oracle.  Returns (errors, contours, rects, external keys)."""
    det, box = h.fit_min_area_rect(img, mode, 1, minLen, lwTresh)
    edges = h.stage(0, 0, "canny")
    if not np.array_equal(edges, cv2.Canny(img, 0, 255)):
        return ["canny differs from cv2.Canny at %d pixels" % int((edges != cv2.Canny(img, 0, 255)).sum())], {}, None, None
    external = _external_keys(cv2, edges) if mode == 0 else None
    rects = h.stage(0, 0, "rects")
    errs, contours, ref_det = _check_rects(rects, h.stage(0, 0, "box"), edges, minLen, lwTresh, external)
    if not np.array_equal(box, h.stage(0, 0, "box")):
        errs.append("lfd_fit_min_area_rect's box_img differs from the box tap")
    if det != ref_det:
        errs.append("detection %s vs %s" % (det, ref_det))
    return errs, contours, rects, external


def _check_counters(h, contours):
    """The device's warp-path and thread-overflow counters of the last call against the restatement."""
    c = h.counters()
    counts = _path_counts(contours)
    warp = sum(v for k, v in counts.items() if k != "thread")
    assert (c["rects_warp_path"], c["rects_thread_overflow"]) == (warp, counts.get("overflow", 0)), (c, counts)


@pytest.mark.gpu
@pytest.mark.parametrize("H,W", list(SIZES))
def test_rects_match_oracle_on_every_path(cv2mod, H, W):
    """Every contour's rectangle bit-identical to the oracle's, every passing box and the box image identical, on the
    images built for each k_rects_warp path, frame edge and size; the device's path counters equal the restatement's."""
    h = _handle(H, W, max_runs=(1 << 22) if H * W > (1 << 22) else 0)
    try:
        for name, img in _images(cv2mod, H, W).items():
            errs, contours, _, _ = _fit(h, cv2mod, img)
            assert not errs, "%s at %dx%d:\n%s" % (name, H, W, "\n".join(errs[:20]))
            counts = _check_coverage(cv2mod, H, W, name, contours)
            _check_counters(h, contours)
            print("%dx%d %s: %s" % (H, W, name, counts))
    finally:
        h.close()


# ---- RETR_EXTERNAL -------------------------------------------------------------------------------------------------
def _img_external(cv2, H, W):
    """Nested filled rings three deep with a blob in the innermost hole; a square whose outline is closed at its
    top-left corner by one diagonal step and a diamond whose outline has diagonal steps only (their insides are holes
    only in 4-connectivity), each with a ring inside; components whose raster-first pixel is in column 0 or row 0; and
    components whose left neighbour's background run is the first or the last run of its row."""
    img = np.zeros((H, W), np.uint8)
    c, R = (W // 4, H // 2), min(H // 2, W // 4) - 16
    t = max(3, R // 8)
    for r in (R, R - 3 * t, R - 6 * t):
        cv2.circle(img, c, r, 255, -1)
        cv2.circle(img, c, r - t, 0, -1)
    cv2.circle(img, c, max(2, R - 8 * t), 255, -1)
    d = min(H, W) // 12
    x0, y0 = 3 * W // 5, H // 5
    img[y0:y0 + 2 * d, x0:x0 + 2 * d] = 255
    img[y0 + d, x0 + d] = 0
    ym = 3 * H // 5
    cv2.fillPoly(img, [np.array([[x0 + d, ym - d], [x0 + 2 * d, ym], [x0 + d, ym + d], [x0, ym]], np.int32)], 255)
    img[ym, x0 + d] = 0
    img[H - 10:H - 4, 0:6] = 255                                  # raster-first pixel in column 0
    img[0:6, 5 * W // 8:5 * W // 8 + 12] = 255                    # ... in row 0
    img[4:12, 4:12] = 255                                         # left neighbour in the row's first background run
    img[H - 24:H - 14, W // 2:W // 2 + 10] = 255
    img[H - 24:H - 14, 7 * W // 8:] = 255                         # top row reaches column W - 1: the row's last run
    return img


def _external_keys(cv2, edges):
    """Raster-first point of each contour cv2.findContours(RETR_EXTERNAL) retrieves."""
    cs, _ = cv2.findContours(edges, cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_NONE)
    keys = set()
    for c in cs:
        p = c.reshape(-1, 2)
        i = np.lexsort((p[:, 0], p[:, 1]))[0]
        keys.add(int(p[i, 1]) * edges.shape[1] + int(p[i, 0]))
    return keys


def _check_external_coverage(cv2, edges, contours):
    H, W = edges.shape
    keys = _external_keys(cv2, edges)
    outer = {key for kind, key in contours if kind == 0}
    assert keys <= outer and len(outer - keys) >= 7           # rings, blob and the rings inside the diagonal outlines
    where = set()
    for key in keys:
        y, x = divmod(key, W)
        if x == 0:
            where.add("column 0")
            continue
        if y == 0:
            where.add("row 0")
        bg = edges[y] == 0
        starts = np.flatnonzero(bg & ~np.concatenate(([False], bg[:-1])))
        i = int(np.searchsorted(starts, x - 1, side="right")) - 1
        if len(starts) > 1:
            where.add("first run" if i == 0 else "last run" if i == len(starts) - 1 else "inner run")
    assert where == {"column 0", "row 0", "first run", "last run", "inner run"}, where
    # some hole is closed only by diagonal steps: its pixels belong to the outside in 8-connectivity
    from scipy import ndimage
    bg8, _ = ndimage.label(edges == 0, structure=np.ones((3, 3)))
    outside = bg8[0][edges[0] == 0][0]
    assert (cr.label_bg4(edges)[bg8 == outside] >= 0).any()
    return keys


@pytest.mark.parametrize("H,W", [(1489, 2048), (256, 332)])
def test_external_image_covers_its_cases(cv2mod, H, W):
    """CPU only: the RETR_EXTERNAL image has the nesting, border and run-position cases it was built for."""
    edges = cv2mod.Canny(_img_external(cv2mod, H, W), 0, 255)
    _check_external_coverage(cv2mod, edges, _contours(edges))


@pytest.mark.gpu
@pytest.mark.parametrize("H,W", [(1489, 2048), (256, 332)])
def test_external_keeps_exactly_cv2s_outer_contours(cv2mod, H, W):
    """contoursMode = 0: the kept (kind 0) rectangles are those of the contours cv2.findContours(RETR_EXTERNAL) retrieves,
    each equal to the oracle's on its component's point set; every other contour's entry is kind 2, none is kind 1."""
    img = _img_external(cv2mod, H, W)
    h = _handle(H, W)
    try:
        errs, contours, rects, keys = _fit(h, cv2mod, img, mode=0)
        assert not errs, "\n".join(errs[:20])
        assert keys == _check_external_coverage(cv2mod, h.stage(0, 0, "canny"), contours)
        assert not (rects["kind"] == 1).any()
        assert (rects["kind"] == 2).sum() == len(contours) - len(keys)
        _check_counters(h, {ck: v for ck, v in contours.items() if ck[0] == 0 and ck[1] in keys})
    finally:
        h.close()


# ---- the multi-frame task list -------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("flags", ["KEEP_TAPS", "KEEP_TAPS|SERIAL_PASSES"])
def test_batch_task_list_across_frames(cv2mod, flags):
    """k_rects_warp bisects one flat task list over the frames of a launch (per-frame contour counts prefix-summed 32
    frames at a time).  40 frames, empty ones in the first, the 32nd and the last slot: every frame's and pass's RECTS and
    BOX taps equal the oracle's on that frame's own CANNY tap with the pass's parameters.  With KEEP_TAPS alone the batch
    runs as two halves of 20 frames; SERIAL_PASSES puts all 40 frames into one launch per pass."""
    from lfd_b200 import _lib, synth
    H, W, n = 600, 1000, 40
    shapes = [b(cv2mod, H, W) for b in (_img_thread, _img_overflow, _img_compact, _img_edges)]
    frames = np.zeros((n, H, W), np.float32)
    for f in range(n):
        if f in (0, 31, n - 1):
            continue
        frames[f], _ = synth.make_frame(7000 + f, n_stars=60 + 5 * f, h=H, w=W)
        frames[f][shapes[f % len(shapes)] > 0] = 1000.0
    params = (rp.DEFAULT_BRIGHT, rp.DEFAULT_DIM)
    h = _lib.Handle(H, W, max_batch=n)
    try:
        h.set_params(dict(params[0]), dict(params[1]))
        fl = 0
        for name in flags.split("|"):
            fl |= getattr(_lib, name)
        h.submit(frames, flags=fl)
        h.wait()
        ncont = []
        for f in range(n):
            for p in (0, 1):
                edges = h.stage(f, p, "canny")
                errs, contours, _ = _check_rects(h.stage(f, p, "rects"), h.stage(f, p, "box"), edges,
                                                 params[p]["minAreaRectMinLen"], params[p]["lwTresh"])
                assert not errs, "frame %d pass %d:\n%s" % (f, p, "\n".join(errs[:20]))
                ncont.append(len(contours))
        assert ncont[0] == ncont[1] == ncont[62] == ncont[63] == ncont[78] == ncont[79] == 0
        assert min(ncont[2:62] + ncont[64:78]) > 0 and sum(ncont) > 2000
    finally:
        h.close()


# ---- contour capacity ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_max_components_at_and_below_the_contour_count(cv2mod):
    """max_components equal to the larger per-kind contour count gives the unconstrained result; one below reports
    LFD_E_CAPACITY, and the next call on the same handle starts clean."""
    from lfd_b200 import _lib
    H, W = 256, 332
    img = _img_thread(cv2mod, H, W)
    edges = cv2mod.Canny(img, 0, 255)
    kinds = [k for k, _, _ in cr.contour_point_sets(edges)]
    mc = max(kinds.count("outer"), kinds.count("hole"))
    out = {}
    for cap in (0, mc):
        h = _handle(H, W, max_components=cap)
        try:
            errs, _, rects, _ = _fit(h, cv2mod, img)
            assert not errs, "max_components %d:\n%s" % (cap, "\n".join(errs[:20]))
            out[cap] = (np.sort(rects, order=["kind", "key"]).tobytes(), h.stage(0, 0, "box"))
        finally:
            h.close()
    assert out[0][0] == out[mc][0] and np.array_equal(out[0][1], out[mc][1])
    h = _handle(H, W, max_components=mc - 1)
    try:
        with pytest.raises(_lib.LfdError) as e:
            h.fit_min_area_rect(img, 1, 1, 0.0, 0.5)
        assert e.value.code == _lib.LFD_E_CAPACITY
        small = _img_overflow(cv2mod, H, W)                     # a handful of contours: the next call is exact
        errs, contours, _, _ = _fit(h, cv2mod, small)
        assert not errs and 0 < len(contours) < mc - 1, errs[:20]
    finally:
        h.close()
