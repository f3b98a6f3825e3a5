"""CPU check of the chord decomposition that k_morph_any evaluates (lfd_b200/csrc/chords.cuh, compiled for the host by
tests/hostchords.cpp): the chords are disjoint, maximal and cover the mask, their count respects the bound the device
buffer is sized by, and the sparse-table evaluation over them (restated in NumPy below, level by level as the kernel
builds it) equals cv2.erode / cv2.dilate bit for bit, with cv2's default anchor and border (out-of-frame samples
ignored)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def hc(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("hc") / "libhostchords.so")
    subprocess.run(["g++", "-O2", "-shared", "-fPIC", "-x", "c++", os.path.join(HERE, "hostchords.cpp"), "-o", out],
                   check=True, stderr=subprocess.DEVNULL)
    return ctypes.CDLL(out)


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def decompose(hc, mask):
    """[(row, start column, length)] in the library's order, and its level count."""
    m = np.ascontiguousarray(np.asarray(mask) != 0, np.uint8)
    kh, kw = m.shape
    rowoff = np.zeros(kh + 1, np.int32)
    code = np.zeros(max(hc.hc_capacity(kh, kw), 1), np.uint32)
    nlev = ctypes.c_int(-1)
    n = hc.hc_decompose(_p(m), kh, kw, _p(rowoff), _p(code), ctypes.byref(nlev))
    assert n == rowoff[kh] <= hc.hc_capacity(kh, kw)
    chords = []
    for i in range(kh):
        for q in code[rowoff[i]:rowoff[i + 1]]:
            q = int(q)
            a, b, k = q & 255, (q >> 8) & 255, (q >> 16) & 15
            L = b - a + (1 << k)
            assert (1 << k) <= L < (2 << k), (a, b, k)
            chords.append((i, a, L))
    return chords, nlev.value


def chord_morph(img, mask, chords, nlev, is_max):
    """cv2.dilate (is_max) / cv2.erode of img over the chords: out(y, x) = op over chords (i, a, L) of
    op(P_k(y + i - ay, x + a - ax), P_k(y + i - ay, x + a - ax + L - 2^k)), P_k the per-row sparse table."""
    kh, kw = np.asarray(mask).shape
    ay, ax = kh // 2, kw // 2
    H, W = img.shape
    ident = 0 if is_max else 255
    op = np.maximum if is_max else np.minimum
    pad = np.full((H + kh, W + 2 * kw), ident, np.uint8)       # rows ay above / kh - ay below, kw columns each side
    pad[ay:ay + H, kw:kw + W] = img
    lv = [pad]
    for k in range(1, nlev):
        s = 1 << (k - 1)
        p = lv[-1]
        q = np.full_like(p, ident)
        q[:, :-s] = op(p[:, :-s], p[:, s:])
        lv.append(q)
    out = np.full((H, W), ident, np.uint8)
    for i, a, L in chords:
        k = L.bit_length() - 1
        assert k < nlev
        c1 = kw + a - ax
        c2 = c1 + L - (1 << k)
        out = op(out, op(lv[k][i:i + H, c1:c1 + W], lv[k][i:i + H, c2:c2 + W]))
    return out


def check_mask(cv2mod, hc, mask, imgs):
    mask = np.ascontiguousarray(np.asarray(mask) != 0, np.uint8)
    kh, kw = mask.shape
    chords, nlev = decompose(hc, mask)
    # disjoint, maximal, and covering the mask
    cover = np.zeros_like(mask, np.int32)
    for i, a, L in chords:
        cover[i, a:a + L] += 1
        assert a == 0 or not mask[i, a - 1]
        assert a + L == kw or not mask[i, a + L]
    assert np.array_equal(cover, mask.astype(np.int32))
    lmax = max(L for _, _, L in chords)
    assert nlev == lmax.bit_length()
    for img in imgs:
        for is_max in (False, True):
            ref = (cv2mod.dilate if is_max else cv2mod.erode)(img, mask)
            got = chord_morph(img, mask, chords, nlev, is_max)
            assert np.array_equal(got, ref), (mask.shape, img.shape, "dilate" if is_max else "erode",
                                              int((got != ref).sum()))


def images(rng, kh, kw):
    """A sparse image a little larger than the element, one smaller than it, and a dense one holding 0 and 255."""
    H, W = max(kh + 11, 24), max(kw + 13, 24)
    sparse = ((rng.random((H, W)) < 0.04) * rng.integers(1, 256, (H, W))).astype(np.uint8)
    small = rng.integers(0, 256, (max(kh // 2, 1), max(kw // 3, 1))).astype(np.uint8)
    dense = rng.choice(np.array([0, 255, 7, 128], np.uint8), (H, W), p=[0.4, 0.3, 0.15, 0.15])
    return [sparse, small, dense]


def ellipse(cv2mod, h, w):
    return cv2mod.getStructuringElement(cv2mod.MORPH_ELLIPSE, (w, h))


def test_limits(hc):
    assert hc.hc_max_side() == 255
    assert hc.hc_capacity(255, 255) == 255 * 128
    # the bound is reached: alternating columns
    m = np.zeros((3, 9), np.uint8)
    m[:, ::2] = 1
    chords, nlev = decompose(hc, m)
    assert len(chords) == hc.hc_capacity(3, 9) and nlev == 1
    chords, nlev = decompose(hc, np.zeros((4, 5), np.uint8))
    assert chords == [] and nlev == 0


@pytest.mark.parametrize("side", [1, 2, 3, 5, 8, 15, 31, 32, 33, 41, 63, 64, 100, 127, 128, 200, 254, 255])
def test_ellipses(cv2mod, hc, side):
    rng = np.random.default_rng(side)
    check_mask(cv2mod, hc, ellipse(cv2mod, side, side), images(rng, side, side))


@pytest.mark.parametrize("hw", [(40, 22), (22, 40), (63, 33), (8, 5), (2, 255), (255, 2), (6, 100)])
def test_uneven_ellipses(cv2mod, hc, hw):
    rng = np.random.default_rng(hw[0] * 1000 + hw[1])
    check_mask(cv2mod, hc, ellipse(cv2mod, *hw), images(rng, *hw))


def _cross(h, w):
    k = np.zeros((h, w), np.uint8)
    k[h // 2, :] = 1
    k[:, w // 2] = 1
    return k


def _ring(cv2mod, n, t):
    k = ellipse(cv2mod, n, n)
    k[t:n - t, t:n - t] &= 1 - ellipse(cv2mod, n - 2 * t, n - 2 * t)
    assert not k[n // 2, n // 2]
    return k


def _off_centre(h, w):
    k = np.zeros((h, w), np.uint8)
    k[0, w - w // 4:] = 1
    return k


@pytest.mark.parametrize("name", ["cross5", "cross33", "cross_even", "ring21", "ring65", "off_centre", "off_centre_big",
                                  "row255", "col255", "row1x7", "col64", "ones64", "ones_even", "single", "corner"])
def test_shapes(cv2mod, hc, name):
    masks = {
        "cross5": lambda: _cross(5, 5), "cross33": lambda: _cross(33, 33), "cross_even": lambda: _cross(10, 26),
        "ring21": lambda: _ring(cv2mod, 21, 3), "ring65": lambda: _ring(cv2mod, 65, 5),
        "off_centre": lambda: _off_centre(9, 40), "off_centre_big": lambda: _off_centre(120, 250),
        "row255": lambda: np.ones((1, 255), np.uint8), "col255": lambda: np.ones((255, 1), np.uint8),
        "row1x7": lambda: np.ones((1, 7), np.uint8), "col64": lambda: np.ones((64, 1), np.uint8),
        "ones64": lambda: np.ones((64, 64), np.uint8), "ones_even": lambda: np.ones((4, 34), np.uint8),
        "single": lambda: np.ones((1, 1), np.uint8),
        "corner": lambda: np.pad(np.ones((1, 1), np.uint8), ((0, 30), (16, 0))),     # one member, top right
    }
    m = masks[name]()
    rng = np.random.default_rng(len(name))
    check_mask(cv2mod, hc, m, images(rng, *m.shape))


@pytest.mark.parametrize("density", [0.1, 0.3, 0.5, 0.7, 0.9])
def test_random_masks(cv2mod, hc, density):
    rng = np.random.default_rng(int(density * 100))
    for shape in ((37, 44), (40, 37), (7, 130), (130, 9), (255, 255)):
        m = (rng.random(shape) < density).astype(np.uint8)
        m[rng.integers(shape[0]), rng.integers(shape[1])] = 1
        check_mask(cv2mod, hc, m, images(rng, *shape)[:2] if shape == (255, 255) else images(rng, *shape))
