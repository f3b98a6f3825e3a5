"""ORACLE (test infrastructure, not product code): NumPy/C restatement of the OpenCV and NumPy
routines on lfd.detecttrails' per-frame path.

Call sites restated (paths under /root/reference/lfd/detecttrails/):
  processfield.py:346,456  cv2.convertScaleAbs   -> convert_scale_abs
  processfield.py:347,457  cv2.equalizeHist      -> equalize_hist / equalize_lut
  processfield.py:354,464,471 cv2.dilate / erode -> morph
  processfield.py:236      cv2.Canny(img,0,255)  -> canny / canny_classes
  processfield.py:241-246  cv2.findContours      -> contour_point_sets (structural equivalent)
  processfield.py:249      cv2.minAreaRect       -> hull + min_area_rect
  processfield.py:259-261  boxPoints/int32/fillPoly -> box_points / fill_poly
  processfield.py:370-371  cv2.HoughLines        -> hough_lines (accumulator exposed)
  detecttrails.py:124      cv2.flip(img, 0)      -> img[::-1]

OpenCV is a third-party dependency absent from /root/reference (setup.py:18-28, unpinned; the
parity target is cv2 4.13.0 as installed).  Everything here is pinned bit-for-bit against that
binary in tests/test_oracle_cv.py.  The heavy loops live in oracle/c/cvrestate.c
(``make -C oracle``).  Only tests/, smoke() and bench.py's CPU-baseline leg may import this.
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def build():
    subprocess.run(["make", "-C", _HERE], check=True, stdout=subprocess.DEVNULL)


def lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(_HERE, "_build", "libcvrestate.so")
        if not os.path.exists(path):
            build()
        _LIB = ctypes.CDLL(path)
        _LIB.orc_hough_lines.restype = ctypes.c_int
        _LIB.orc_hull.restype = ctypes.c_int
        _LIB.orc_clip_line.restype = ctypes.c_int
    return _LIB


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


# ----------------------------------------------------------------------------------------------
def clip_bright(img):
    """processfield.py:342  img[img < 0] = 0 (NaN untouched)."""
    out = img.copy()
    out[out < 0] = 0
    return out


def clip_dim(img, minFlux, addFlux):
    """processfield.py:453-454 on an array bright has already clipped."""
    out = img.copy()
    out[out < minFlux] = 0
    out[out > 0] += addFlux
    return out


def convert_scale_abs(img):
    """u8 = saturate(rint(|v|)), half-to-even; NaN/inf/|v| >= 2**31 -> 0 (x86 cvtps2dq indefinite)."""
    a = np.abs(img.astype(np.float32))
    r = np.rint(a)
    bad = ~np.isfinite(a) | (a >= np.float32(2147483648.0))
    r = np.where(bad, 0, np.minimum(r, 255))
    return r.astype(np.uint8)


def equalize_lut(hist):
    """The 256-entry LUT cv2.equalizeHist applies, from a 256-bin histogram (int)."""
    hist = np.asarray(hist, np.int64)
    total = int(hist.sum())
    nz = np.nonzero(hist)[0]
    lut = np.arange(256, dtype=np.uint8)
    if len(nz) == 0:
        return lut
    i0 = int(nz[0])
    if hist[i0] == total:
        return lut  # constant image: dst = src
    scale = np.float32(255.0) / np.float32(total - hist[i0])
    s = np.cumsum(hist[i0 + 1:])
    vals = np.rint(s.astype(np.float32) * scale)
    lut = np.zeros(256, np.uint8)
    lut[i0 + 1:] = np.clip(vals, 0, 255).astype(np.uint8)
    return lut


def equalize_hist(gray):
    hist = np.bincount(gray.ravel(), minlength=256)
    return equalize_lut(hist)[gray]


def morph(img, kernel, op):
    """erode ('min') / dilate ('max') with an arbitrary uint8 kernel; anchor (kw//2, kh//2);
    out-of-frame samples ignored."""
    kernel = np.asarray(kernel)
    kh, kw = kernel.shape
    ay, ax = kh // 2, kw // 2
    H, W = img.shape
    fill = 255 if op == "min" else 0
    pad = np.full((H + kh, W + kw), fill, np.uint8)
    pad[ay:ay + H, ax:ax + W] = img
    out = np.full((H, W), fill, np.uint8)
    f = np.minimum if op == "min" else np.maximum
    for dy in range(kh):
        for dx in range(kw):
            if kernel[dy, dx]:
                out = f(out, pad[dy:dy + H, dx:dx + W])
    return out


def canny_classes(img, low=0, high=255):
    """(cls, mag): cls 0 none / 1 weak / 2 strong after NMS."""
    img = np.ascontiguousarray(img, np.uint8)
    H, W = img.shape
    cls = np.empty((H, W), np.uint8)
    mag = np.empty((H, W), np.int32)
    lib().orc_canny_classes(_p(img), H, W, int(low), int(high), _p(cls), _p(mag))
    return cls, mag


def canny(img, low=0, high=255):
    cls, _ = canny_classes(img, low, high)
    H, W = cls.shape
    edges = np.empty((H, W), np.uint8)
    lib().orc_canny_hysteresis(_p(cls), H, W, _p(edges))
    return edges


def label_fg8(img):
    img = np.ascontiguousarray(img, np.uint8)
    lab = np.empty(img.shape, np.int32)
    lib().orc_label_fg8(_p(img), img.shape[0], img.shape[1], _p(lab))
    return lab


def label_bg4(img):
    img = np.ascontiguousarray(img, np.uint8)
    lab = np.empty(img.shape, np.int32)
    lib().orc_label_bg4(_p(img), img.shape[0], img.shape[1], _p(lab))
    return lab


def contour_point_sets(edges):
    """Structural equivalent of findContours(RETR_LIST, CHAIN_APPROX_NONE) (SURVEY.md 9.5):
    one point set per 8-connected foreground component (outer border) and one per 4-connected
    background component that does not reach the frame border (hole border = foreground pixels
    4-adjacent to the hole).  Returns list of (kind, key, points int32 (n,2) as x,y)."""
    H, W = edges.shape
    fg = label_fg8(edges)
    bg = label_bg4(edges)
    out = []
    ys, xs = np.nonzero(fg >= 0)
    if len(ys) == 0:
        return out          # no edge pixel: no contour, and no hole either
    labs = fg[ys, xs]
    order = np.argsort(labs, kind="stable")
    ys, xs, labs = ys[order], xs[order], labs[order]
    cuts = np.flatnonzero(np.diff(labs)) + 1
    for yy, xx, ll in zip(np.split(ys, cuts), np.split(xs, cuts), np.split(labs, cuts)):
        out.append(("outer", int(ll[0]), np.stack([xx, yy], 1).astype(np.int32)))
    hy, hx = np.nonzero(bg >= 0)
    if len(hy):
        hl = bg[hy, hx]
        pts_l, pts_x, pts_y = [], [], []
        for dy, dx in ((0, -1), (0, 1), (-1, 0), (1, 0)):
            ny, nx = hy + dy, hx + dx  # holes never touch the border, so neighbours are in range
            m = edges[ny, nx] != 0
            pts_l.append(hl[m]); pts_x.append(nx[m]); pts_y.append(ny[m])
        pl, px, py = np.concatenate(pts_l), np.concatenate(pts_x), np.concatenate(pts_y)
        order = np.argsort(pl, kind="stable")
        pl, px, py = pl[order], px[order], py[order]
        cuts = np.flatnonzero(np.diff(pl)) + 1
        for xx, yy, ll in zip(np.split(px, cuts), np.split(py, cuts), np.split(pl, cuts)):
            out.append(("hole", int(ll[0]), np.stack([xx, yy], 1).astype(np.int32)))
    return out


def hull(points):
    """Convex hull (float32 (m,2)) of int points in cv2.convexHull(clockwise=False) order, started
    at the lexicographic maximum (cv2's own cyclic shift depends on the contour's traversal order;
    see DESIGN.md 'hull start vertex')."""
    pts = np.ascontiguousarray(points, np.int32).reshape(-1, 2)
    out = np.empty((len(pts) + 1, 2), np.float32)
    m = lib().orc_hull(_p(pts), len(pts), _p(out))
    return out[:m].copy()


def min_area_rect(hull_pts):
    """((cx, cy), (w, h), angle) as python floats of float32 values, like cv2.minAreaRect."""
    h = np.ascontiguousarray(hull_pts, np.float32).reshape(-1, 2)
    out = np.zeros(5, np.float32)
    lib().orc_min_area_rect(_p(h), len(h), _p(out))
    return ((float(out[0]), float(out[1])), (float(out[2]), float(out[3])), float(out[4]))


def box_points(rect):
    r = np.array([rect[0][0], rect[0][1], rect[1][0], rect[1][1], rect[2]], np.float32)
    out = np.empty(8, np.float32)
    lib().orc_box_points(_p(r), _p(out))
    return out.reshape(4, 2)


def clip_line(W, H, p1, p2):
    buf = np.array([p1[0], p1[1], p2[0], p2[1]], np.int64)
    ok = lib().orc_clip_line(int(W), int(H), _p(buf))
    return bool(ok), (int(buf[0]), int(buf[1])), (int(buf[2]), int(buf[3]))


def line8(img, p1, p2, val=255):
    lib().orc_line8(_p(img), img.shape[0], img.shape[1], int(p1[0]), int(p1[1]), int(p2[0]), int(p2[1]), int(val))
    return img


def fill_poly(img, poly, val=255):
    v = np.ascontiguousarray(poly, np.int32).reshape(-1, 2)
    lib().orc_fill_poly(_p(img), img.shape[0], img.shape[1], _p(v), len(v), int(val))
    return img


def hough_dims(H, W, rho, theta):
    na, nr = ctypes.c_int(), ctypes.c_int()
    lib().orc_hough_dims(int(H), int(W), ctypes.c_double(rho), ctypes.c_double(theta), ctypes.byref(na), ctypes.byref(nr))
    return na.value, nr.value


def hough_lines(img, rho, theta, threshold):
    """Returns (lines (n,1,2) float32 or None, accumulator (numangle+2, numrho+2) int32, votes)."""
    img = np.ascontiguousarray(img, np.uint8)
    H, W = img.shape
    na, nr = hough_dims(H, W, rho, theta)
    accum = np.empty((na + 2, nr + 2), np.int32)
    cap = na * nr
    lines = np.empty((cap, 2), np.float32)
    votes = np.empty(cap, np.int32)
    n = lib().orc_hough_lines(_p(img), H, W, ctypes.c_double(rho), ctypes.c_double(theta), int(threshold),
                              _p(accum), _p(lines), _p(votes), cap)
    if n == 0:
        return None, accum, votes[:0]
    return lines[:n].reshape(n, 1, 2).copy(), accum, votes[:n].copy()


def rects_and_box(edges, minAreaRectMinLen, lwTresh):
    """fit_minAreaRect's loop (processfield.py:248-261) over the structural contour sets."""
    H, W = edges.shape
    box_img = np.zeros((H, W), np.uint8)
    rects, passing = [], []
    for kind, key, pts in contour_point_sets(edges):
        r = min_area_rect(hull(pts))
        rects.append((kind, key, r))
        w, h = r[1]
        length, width = (w, h) if w > h else (h, w)
        if length > minAreaRectMinLen and width > minAreaRectMinLen and length / width > lwTresh:
            box = box_points(r).astype(np.int32)
            fill_poly(box_img, box, 255)
            passing.append((kind, key, r, box))
    return rects, passing, box_img
