"""ctypes binding of liblfd_b200.so (include/lfd_b200.h).  No torch, no cv2, no CPU fallback:
if the CUDA library is missing or no GPU is present the import of the library / creation of a
handle raises and the caller sees it."""
import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
LIB_PATH = os.environ.get("LFD_B200_LIB") or os.path.join(HERE, "liblfd_b200.so")     # env override: A/B builds in profiles/lab
SRC = os.path.join(HERE, "csrc", "lfd_b200.cu")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-fmad=false", "-std=c++17",
              "-Xcompiler", "-fPIC,-Winit-self,-Wuninitialized", "-shared"]

LFD_OK, LFD_E_ARG, LFD_E_CUDA, LFD_E_UNSUPPORTED, LFD_E_CAPACITY, LFD_E_STATE = 0, -1, -2, -3, -4, -5
FRAME_OVERFLOW, FRAME_NO_LINES_EQU, FRAME_NO_LINES_BOX = 1, 2, 4
PASS_BRIGHT, PASS_DIM = 0, 1
INPUT_NATIVE, INPUT_BIGENDIAN, KEEP_TAPS, FULL_LINES, SERIAL_PASSES, KERNEL_TIMES = 0, 1, 2, 4, 8, 16
MAX_SET_LINES = 16

STAGES = {"mask": 0, "gray": 1, "equ": 2, "eroded": 3, "morph": 4, "canny": 5, "box": 6, "hist": 7, "lut": 8,
          "nms": 9, "fg_labels": 10, "bg_labels": 11, "rects": 12, "accum_equ": 13, "accum_box": 14,
          "lines_equ": 15, "lines_box": 16, "clipped": 17, "input": 18, "rect_screen": 19}
MAX_INJECT_TRAILS = 16
TRAIL_DTYPE = np.dtype([("x0", "<f4"), ("y0", "<f4"), ("x1", "<f4"), ("y1", "<f4"), ("sigma", "<f4"), ("peak", "<f4")])
MAX_TABLE_SAMPLES, MAX_TRAIL_TABLES = 4096, 4096
TABLE_DTYPE = np.dtype([("offset", "<i4"), ("n", "<i4"), ("lo", "<f4"), ("hi", "<f4")])
SHAPE_DTYPE = np.dtype([("profile", "<i4"), ("lightcurve", "<i4")])


class PassParams(ctypes.Structure):
    _fields_ = [("lwTresh", ctypes.c_double), ("thetaTresh", ctypes.c_double), ("lineSetTresh", ctypes.c_double),
                ("dro", ctypes.c_double), ("minAreaRectMinLen", ctypes.c_double), ("houghMethod", ctypes.c_double),
                ("minFlux", ctypes.c_double), ("addFlux", ctypes.c_double), ("nlinesInSet", ctypes.c_int32),
                ("contoursMode", ctypes.c_int32), ("contoursMethod", ctypes.c_int32),
                ("erode_h", ctypes.c_int32), ("erode_w", ctypes.c_int32),
                ("dilate_h", ctypes.c_int32), ("dilate_w", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class Params(ctypes.Structure):
    _fields_ = [("bright", PassParams), ("dim", PassParams)]


class Result(ctypes.Structure):
    _fields_ = [("detected", ctypes.c_int32), ("pass_", ctypes.c_int32), ("status", ctypes.c_int32),
                ("rect_detection", ctypes.c_int32 * 2), ("n_lines_equ", ctypes.c_int32 * 2),
                ("n_lines_box", ctypes.c_int32 * 2), ("rejected", ctypes.c_int32 * 2),
                ("rho", ctypes.c_float), ("theta", ctypes.c_float),
                ("top_equ", ((ctypes.c_float * 2) * MAX_SET_LINES) * 2),
                ("top_box", ((ctypes.c_float * 2) * MAX_SET_LINES) * 2)]


RECT_DTYPE = np.dtype([("cx", "<f4"), ("cy", "<f4"), ("w", "<f4"), ("h", "<f4"), ("angle", "<f4"),
                       ("kind", "<i4"), ("key", "<i4"), ("passed", "<i4"), ("box", "<i4", (8,))])


class Config(ctypes.Structure):
    _fields_ = [("max_runs", ctypes.c_int32), ("max_components", ctypes.c_int32), ("max_star_rects", ctypes.c_int32),
                ("max_lines", ctypes.c_int32), ("reserved", ctypes.c_int32 * 4)]


class LfdError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("lfd_b200 error %d: %s" % (code, msg))
        self.code = code


class UnsupportedParameter(LfdError):
    pass


def build(force=False, verbose=False):
    """Compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    srcs = [os.path.join(HERE, "csrc", f) for f in os.listdir(os.path.join(HERE, "csrc"))]
    srcs.append(os.path.join(ROOT, "include", "lfd_b200.h"))
    if not force and os.path.exists(LIB_PATH):
        if os.path.getmtime(LIB_PATH) >= max(os.path.getmtime(s) for s in srcs):
            return LIB_PATH
    cmd = ["nvcc"] + NVCC_FLAGS + [SRC, "-o", LIB_PATH]
    if verbose:
        print(" ".join(cmd))
    subprocess.run(cmd, check=True)
    return LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("liblfd_b200.so is not built (run `python -c 'import __graft_entry__ as g; g.build()'`); "
                              "there is no CPU fallback")
        L = ctypes.CDLL(LIB_PATH)
        L.lfd_last_error.restype = ctypes.c_char_p
        L.lfd_last_error.argtypes = [ctypes.c_void_p]
        L.lfd_timing_name.restype = ctypes.c_char_p
        L.lfd_kernel_launches.restype = ctypes.c_int64
        L.lfd_kernel_launches.argtypes = [ctypes.c_void_p]
        L.lfd_create_ex.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                                    ctypes.POINTER(ctypes.c_void_p)]
        L.lfd_destroy.argtypes = [ctypes.c_void_p]
        L.lfd_set_params.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        L.lfd_set_h2d_gate.argtypes = [ctypes.c_void_p, ctypes.c_char_p]
        L.lfd_set_kernels.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
                                      ctypes.c_void_p, ctypes.c_int, ctypes.c_int]
        L.lfd_host_frames.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p)]
        L.lfd_submit.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]
        L.lfd_upload.argtypes = L.lfd_submit.argtypes
        L.lfd_run_resident.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int]
        L.lfd_wait.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        L.lfd_run_pass.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
        L.lfd_blot.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]
        L.lfd_get_stage.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t]
        L.lfd_get_stage_count.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_int)]
        L.lfd_hough_dims.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_double,
                                     ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]
        L.lfd_hough_lines.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_double,
                                      ctypes.c_double, ctypes.c_int, ctypes.c_void_p, ctypes.c_int,
                                      ctypes.POINTER(ctypes.c_int), ctypes.c_void_p]
        L.lfd_canny.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
        L.lfd_smem_atomic_peak.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_double)]
        L.lfd_fit_min_area_rect.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_double,
                                            ctypes.c_double, ctypes.c_void_p, ctypes.POINTER(ctypes.c_int)]
        L.lfd_get_timings.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_int)]
        L.lfd_get_counters.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]
        L.lfd_get_kernel_times.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(ctypes.c_int),
                                           ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_int)]
        L.lfd_timer_mark.argtypes = [ctypes.c_void_p, ctypes.c_int]
        L.lfd_timer_elapsed.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_float)]
        L.lfd_fits_load_frame.argtypes = [ctypes.c_char_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
                                          ctypes.POINTER(ctypes.c_char_p), ctypes.c_int, ctypes.c_char_p]
        L.lfd_catalog_rects.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double,
                                        ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_longlong,
                                        ctypes.c_double, ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_int)]
        L.lfd_ingest_batch.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_char_p),
                                       ctypes.POINTER(ctypes.c_char_p), ctypes.c_void_p, ctypes.c_void_p, ctypes.c_double,
                                       ctypes.c_double, ctypes.c_double, ctypes.c_longlong, ctypes.c_double,
                                       ctypes.POINTER(ctypes.c_char_p), ctypes.c_int, ctypes.c_char_p, ctypes.c_void_p, ctypes.c_int,
                                       ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]
        for sym in ("lfd_set_base", "lfd_submit_injected", "lfd_set_trail_tables", "lfd_submit_injected_shaped",
                    "lfd_capture_bases"):
            # added within ABI version 1: a stale build lacks them
            if not hasattr(L, sym):
                raise ImportError("liblfd_b200.so predates %s: rebuild it (`python -c 'import __graft_entry__ as g; g.build()'`)" % sym)
        L.lfd_set_base.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
        L.lfd_submit_injected.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                          ctypes.c_int]
        L.lfd_set_trail_tables.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
        L.lfd_submit_injected_shaped.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                                 ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]
        L.lfd_capture_bases.argtypes = [ctypes.c_void_p]
        if L.lfd_abi_version() != 1:
            raise ImportError("liblfd_b200.so ABI mismatch")
        _lib = L
    return _lib


# ---- host-side ingest in native code (include/lfd_b200.h: lfd_fits_load_frame, lfd_catalog_rects) ------------------
HEADER_KEYS = ("TAI", "CRPIX1", "CRPIX2", "CRVAL1", "CRVAL2", "CD1_1", "CD1_2", "CD2_1", "CD2_2")   # detecttrails.py:115-117
_KEYS_C = (ctypes.c_char_p * len(HEADER_KEYS))(*[k.encode() for k in HEADER_KEYS])
_BANDS = "ugriz"


def fits_load_frame(path, slot):
    """Raw big-endian payload of a plain float32 frame file -> ``slot`` (a C-contiguous (H, W) 4-byte array, e.g. a row
    of a handle's pinned staging); returns {key: raw card value text} for HEADER_KEYS, or None when the file is not
    of that plain kind (the caller then uses the general Python reader).  The GIL is released for the whole call."""
    vals = ctypes.create_string_buffer(72 * len(HEADER_KEYS))
    rc = lib().lfd_fits_load_frame(os.fsencode(path), slot.ctypes.data_as(ctypes.c_void_p), slot.shape[0], slot.shape[1],
                                   _KEYS_C, len(HEADER_KEYS), vals)
    if rc != LFD_OK:
        return None
    raw = vals.raw
    return {k: raw[72 * i:72 * i + 72].split(b"\0", 1)[0].decode("ascii", errors="replace") for i, k in enumerate(HEADER_KEYS)}


def catalog_rects(path, _filter, shape, defaultxy, filter_caps, maxxy, pixscale, magcount, maxmagdiff, debug=False):
    """Blot rectangles of one photoObj file, filter and slice rules of ``removestars.star_rects`` in native code; None
    when the table is not the plain photoObj layout or needs the Python path's exceptions (non-finite values)."""
    try:
        band = _BANDS.index(_filter)
        args = (float(filter_caps[_filter]), float(maxmagdiff), float(magcount), float(pixscale), int(defaultxy), float(maxxy))
        cap = max(os.path.getsize(path) // 88 + 1, 1)          # a row holds at least the six columns (4 x 20 + 2 x 4 bytes)
    except (ValueError, TypeError, KeyError, OverflowError, OSError):
        return None
    out = np.empty((cap, 4), np.int32)
    n = ctypes.c_int(0)
    rc = lib().lfd_catalog_rects(os.fsencode(path), band, int(shape[0]), int(shape[1]), args[0], args[1], args[2], args[3],
                                 args[4], args[5], out.ctypes.data_as(ctypes.c_void_p), cap, ctypes.byref(n))
    if rc != LFD_OK:
        return None
    return out[:n.value].copy() if n.value * 4 < cap else out[:n.value]


class BatchIngest:
    """Result of ``ingest_batch``: per-frame status of the frame / catalog reader (0 = done natively), the raw header
    card texts, and the blot rectangles (``rects[i, :n_rects[i]]``)."""
    __slots__ = ("status_frame", "status_cat", "values", "rects", "n_rects", "nkeys")

    def header(self, i):
        raw = self.values.raw
        base = 72 * self.nkeys * i
        return {k: raw[base + 72 * j:base + 72 * j + 72].split(b"\0", 1)[0].decode("ascii", errors="replace")
                for j, k in enumerate(HEADER_KEYS)}


def ingest_batch(staging, frame_paths, cat_paths, filters, defaultxy, filter_caps, maxxy, pixscale, magcount, maxmagdiff,
                 debug=False, max_rects=8192, nthreads=0):
    """lfd_ingest_batch: frames into ``staging[i]`` (rows of a handle's pinned buffer viewed as 4-byte items, shape
    (B, H, W)), catalogs into rectangles, on native threads with the GIL released.  Returns a BatchIngest, or None when
    the parameters cannot be expressed natively (the caller then loads frame by frame)."""
    n = len(frame_paths)
    try:
        bands = np.array([_BANDS.index(f) for f in filters], np.int32)
        caps = np.array([float(filter_caps[b]) for b in _BANDS], np.float64)
        args = (float(maxmagdiff), float(magcount), float(pixscale), int(defaultxy), float(maxxy))
    except (ValueError, TypeError, KeyError, OverflowError):
        return None
    out = BatchIngest()
    out.nkeys = len(HEADER_KEYS)
    out.values = ctypes.create_string_buffer(72 * out.nkeys * max(n, 1))
    out.rects = np.empty((max(n, 1), max_rects, 4), np.int32)
    out.n_rects = np.zeros(max(n, 1), np.int32)
    out.status_frame = np.full(max(n, 1), LFD_E_ARG, np.int32)
    out.status_cat = np.full(max(n, 1), LFD_E_ARG, np.int32)
    fp = (ctypes.c_char_p * max(n, 1))(*[os.fsencode(p) if p else None for p in frame_paths])
    cp = (ctypes.c_char_p * max(n, 1))(*[os.fsencode(p) if p else None for p in cat_paths])
    rc = lib().lfd_ingest_batch(staging.ctypes.data_as(ctypes.c_void_p), int(staging.shape[1]), int(staging.shape[2]), n, fp, cp,
                                bands.ctypes.data_as(ctypes.c_void_p), caps.ctypes.data_as(ctypes.c_void_p), args[0], args[1], args[2],
                                args[3], args[4], _KEYS_C, out.nkeys, out.values, out.rects.ctypes.data_as(ctypes.c_void_p), max_rects,
                                out.n_rects.ctypes.data_as(ctypes.c_void_p), out.status_frame.ctypes.data_as(ctypes.c_void_p),
                                out.status_cat.ctypes.data_as(ctypes.c_void_p), int(nthreads))
    return out if rc == LFD_OK else None


def _kernel_hw(kernel, name):
    if kernel is None:
        return 0, 0
    k = np.asarray(kernel)
    if k.ndim != 2 or k.size == 0:
        raise ValueError("%s must be a 2-D array" % name)
    return int(k.shape[0]), int(k.shape[1])


def _all_ones(kernel):
    return kernel is None or bool(np.all(np.asarray(kernel) != 0))


def pass_params(d, dim):
    """params_bright / params_dim dict (reference keys, detecttrails.py:202-230) -> PassParams."""
    p = PassParams()
    p.lwTresh = float(d["lwTresh"])
    p.thetaTresh = float(d["thetaTresh"])
    p.lineSetTresh = float(d["lineSetTresh"])
    p.dro = float(d["dro"])
    p.minAreaRectMinLen = float(d["minAreaRectMinLen"])
    p.houghMethod = float(d["houghMethod"])
    p.minFlux = float(d.get("minFlux", 0.0)) if dim else 0.0
    p.addFlux = float(d.get("addFlux", 0.0)) if dim else 0.0
    p.nlinesInSet = int(d["nlinesInSet"])
    p.contoursMode = int(d["contoursMode"])
    p.contoursMethod = int(d["contoursMethod"])
    p.erode_h, p.erode_w = _kernel_hw(d.get("erodeKernel"), "erodeKernel") if dim else (0, 0)
    p.dilate_h, p.dilate_w = _kernel_hw(d["dilateKernel"], "dilateKernel")
    return p


class Handle:
    """One GPU worker: owns device buffers for `max_batch` frames of (height, width)."""

    def __init__(self, height, width, max_batch=1, device=0, max_runs=0, max_components=0, max_star_rects=0, max_lines=0):
        L = lib()
        self._L = L
        self.h = ctypes.c_void_p()
        cfg = Config(max_runs, max_components, max_star_rects, max_lines)
        rc = L.lfd_create_ex(device, max_batch, height, width, ctypes.byref(cfg), ctypes.byref(self.h))
        if rc != LFD_OK:
            self.h = None
            raise LfdError(rc, (L.lfd_last_error(None) or b"").decode())
        self.H, self.W, self.B, self.device = height, width, max_batch, device
        self._params_key = None
        hp = ctypes.c_void_p()
        self._ck(L.lfd_host_frames(self.h, ctypes.byref(hp)))
        buf = (ctypes.c_float * (max_batch * height * width)).from_address(hp.value)
        self.host_frames = np.frombuffer(buf, dtype=np.float32).reshape(max_batch, height, width)
        self._results = (Result * max_batch)()

    def _ck(self, rc):
        if rc != LFD_OK:
            msg = (self._L.lfd_last_error(self.h) or b"").decode()
            raise (UnsupportedParameter if rc == LFD_E_UNSUPPORTED else LfdError)(rc, msg)

    def close(self):
        if getattr(self, "h", None):
            self.host_frames = None
            self._L.lfd_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_h2d_gate(self, lock_path):
        """Share a host->device copy slot (an advisory lock file) with the other ranks behind the same host bridge;
        None removes the gate (include/lfd_b200.h: lfd_set_h2d_gate)."""
        self._ck(self._L.lfd_set_h2d_gate(self.h, os.fsencode(lock_path) if lock_path else None))

    def set_params(self, params_bright, params_dim):
        key = repr((sorted((k, np.asarray(v).tolist()) for k, v in params_bright.items() if k != "debug"),
                    sorted((k, np.asarray(v).tolist()) for k, v in params_dim.items() if k != "debug")))
        if key == self._params_key:
            return
        P = Params(pass_params(params_bright, False), pass_params(params_dim, True))
        # structuring elements that are not all-ones rectangles go through lfd_set_kernels; the rectangle sizes in
        # the params struct are then placeholders (1x1) so that the rectangle path's halo limits do not apply
        special = []
        for pass_, (dct, pp) in enumerate(((params_bright, P.bright), (params_dim, P.dim))):
            ek = dct.get("erodeKernel") if pass_ == 1 else None
            dk = dct["dilateKernel"]
            eh, ew = _kernel_hw(ek, "erodeKernel")
            dh, dw = _kernel_hw(dk, "dilateKernel")
            # the rectangle kernels stage a 16-row / 12-column halo; wider all-ones rectangles take the general path too
            too_wide = (eh // 2 + dh // 2 > 16) or (ew // 2 + dw // 2 > 11)
            if not (_all_ones(ek) and _all_ones(dk)) or too_wide:
                special.append((pass_, None if ek is None else np.ascontiguousarray(np.asarray(ek) != 0, np.uint8),
                                np.ascontiguousarray(np.asarray(dk) != 0, np.uint8)))
                pp.dilate_h = pp.dilate_w = 1
                if pass_ == 1 and ek is not None:
                    pp.erode_h = pp.erode_w = 1
        self._ck(self._L.lfd_set_params(self.h, ctypes.byref(P)))
        for pass_, ek, dk in special:
            self._ck(self._L.lfd_set_kernels(self.h, pass_, None if ek is None else ek.ctypes.data_as(ctypes.c_void_p),
                                             0 if ek is None else ek.shape[0], 0 if ek is None else ek.shape[1],
                                             dk.ctypes.data_as(ctypes.c_void_p), dk.shape[0], dk.shape[1]))
        self._params_key = key

    @staticmethod
    def _rects_arrays(rects_per_frame):
        if rects_per_frame is None:
            return None, None, None, None
        offs = np.zeros(len(rects_per_frame) + 1, np.int32)
        for i, r in enumerate(rects_per_frame):
            offs[i + 1] = offs[i] + len(r)
        flat = np.zeros((max(int(offs[-1]), 1), 4), np.int32)
        if offs[-1]:
            flat[:offs[-1]] = np.concatenate([np.asarray(r, np.int32).reshape(-1, 4) for r in rects_per_frame if len(r)])
        return flat, offs, flat.ctypes.data_as(ctypes.c_void_p), offs.ctypes.data_as(ctypes.c_void_p)

    def submit(self, frames, rects_per_frame=None, flags=0):
        """frames: (n, H, W) float32 C-contiguous host array, or an int n to use self.host_frames[:n]."""
        if isinstance(frames, (int, np.integer)):
            n, ptr = int(frames), None
        else:
            frames = np.ascontiguousarray(frames, dtype=np.float32 if not (flags & INPUT_BIGENDIAN) else frames.dtype)
            n, ptr = frames.shape[0], frames.ctypes.data_as(ctypes.c_void_p)
        self._keep = (frames, self._rects_arrays(rects_per_frame))
        _, _, rp, op = self._keep[1]
        self._ck(self._L.lfd_submit(self.h, ptr, n, rp, op, flags))
        self._n = n

    def upload(self, frames, rects_per_frame=None, flags=0):
        if isinstance(frames, (int, np.integer)):
            n, ptr = int(frames), None
        else:
            frames = np.ascontiguousarray(frames)
            n, ptr = frames.shape[0], frames.ctypes.data_as(ctypes.c_void_p)
        keep = self._rects_arrays(rects_per_frame)
        self._ck(self._L.lfd_upload(self.h, ptr, n, keep[2], keep[3], flags))
        self._ck(self._L.lfd_run_resident(self.h, n, flags))   # also drains the copy before buffers go away
        self._n = n
        return self.wait()

    def run_resident(self, n, flags=0):
        self._ck(self._L.lfd_run_resident(self.h, n, flags))
        self._n = n

    def wait(self):
        self._ck(self._L.lfd_wait(self.h, ctypes.byref(self._results)))
        self._keep = None
        return [self._results[i] for i in range(self._n)]

    def wait_array(self):
        """lfd_wait, results as a NumPy structured array (a copy; fields named like lfd_result) for vectorised decoding."""
        self._ck(self._L.lfd_wait(self.h, ctypes.byref(self._results)))
        self._keep = None
        return np.frombuffer(self._results, dtype=np.dtype(Result), count=self._n).copy()

    def set_base(self, frames, rects_per_frame=None):
        """Upload (n_base, H, W) native-order, un-flipped float32 frames once as injection bases, with their star
        rectangles (lfd_submit's convention); a second call replaces them (include/lfd_b200.h: lfd_set_base)."""
        frames = np.ascontiguousarray(frames, dtype=np.float32)
        if frames.ndim != 3 or frames.shape[1:] != (self.H, self.W):
            raise ValueError("frames must have shape (n, %d, %d)" % (self.H, self.W))
        _flat, _offs, rp, op = self._rects_arrays(rects_per_frame)
        self._ck(self._L.lfd_set_base(self.h, frames.ctypes.data_as(ctypes.c_void_p), frames.shape[0], rp, op))

    def capture_bases(self):
        """Make the frames of the last collected whole-frame batch the injection bases (base b = slot b, native order,
        with the batch's star rectangles), without any host<->device copy (include/lfd_b200.h: lfd_capture_bases)."""
        self._ck(self._L.lfd_capture_bases(self.h))

    def set_trail_tables(self, tables):
        """Upload the pool of tabulated trail shapes, a list of ``(lo, hi, samples)`` (``samples`` evenly spaced on
        [lo, hi]); a trail dict's ``"profile"`` / ``"lightcurve"`` keys index it.  A second call replaces the pool
        (include/lfd_b200.h: lfd_set_trail_tables, lfd_table)."""
        arrs = [np.asarray(smp, np.float32).ravel() for _lo, _hi, smp in tables]
        tab = np.zeros(len(arrs), TABLE_DTYPE)
        off = 0
        for i, ((lo, hi, _smp), a) in enumerate(zip(tables, arrs)):
            tab[i] = (off, len(a), lo, hi)
            off += len(a)
        pool = np.ascontiguousarray(np.concatenate(arrs) if arrs else np.zeros(0, np.float32))
        self._ck(self._L.lfd_set_trail_tables(self.h, pool.ctypes.data_as(ctypes.c_void_p), len(pool),
                                              tab.ctypes.data_as(ctypes.c_void_p), len(tab)))

    @staticmethod
    def trails_array(trails):
        """Trails as synth's dicts {p0: (x, y), p1: (x, y), sigma, peak} -> a TRAIL_DTYPE array (float32 fields).  A
        trail with a tabulated ``"profile"`` may omit ``sigma`` (NaN here)."""
        out = np.zeros(len(trails), TRAIL_DTYPE)
        for i, t in enumerate(trails):
            sigma = t["sigma"] if t.get("profile", -1) < 0 else t.get("sigma", np.nan)
            out[i] = (t["p0"][0], t["p0"][1], t["p1"][0], t["p1"][1], sigma, t["peak"])
        return out

    def submit_injected(self, base_index, trails_per_slot=None, flags=0):
        """Run slot f on base base_index[f] plus the trails trails_per_slot[f] (synth's dicts), added on the device;
        collect with wait() (include/lfd_b200.h: lfd_submit_injected).  When a trail has an integer ``"profile"`` or
        ``"lightcurve"`` key (an index into set_trail_tables' pool, -1 = Gaussian / constant) the batch goes through
        lfd_submit_injected_shaped."""
        bidx = np.ascontiguousarray(base_index, np.int32)
        n = len(bidx)
        tp, op = None, None
        if trails_per_slot is not None:
            if len(trails_per_slot) != n:
                raise ValueError("trails_per_slot must have one entry per slot")
            offs = np.zeros(n + 1, np.int32)
            for i, ts in enumerate(trails_per_slot):
                offs[i + 1] = offs[i] + len(ts)
            arr = np.zeros(max(int(offs[-1]), 1), TRAIL_DTYPE)
            if offs[-1]:
                arr[:offs[-1]] = np.concatenate([self.trails_array(ts) for ts in trails_per_slot if len(ts)])
            tp, op = arr.ctypes.data_as(ctypes.c_void_p), offs.ctypes.data_as(ctypes.c_void_p)
            flat = [t for ts in trails_per_slot for t in ts]
            if any("profile" in t or "lightcurve" in t for t in flat):
                shapes = np.array([(t.get("profile", -1), t.get("lightcurve", -1)) for t in flat], SHAPE_DTYPE)
                self._ck(self._L.lfd_submit_injected_shaped(self.h, n, bidx.ctypes.data_as(ctypes.c_void_p), tp,
                                                            shapes.ctypes.data_as(ctypes.c_void_p), op, flags))
                self._n = n
                return
        self._ck(self._L.lfd_submit_injected(self.h, n, bidx.ctypes.data_as(ctypes.c_void_p), tp, op, flags))
        self._n = n

    def run_pass(self, pass_, img, flags=0, writeback=True):
        if img.dtype != np.float32 or not img.flags["C_CONTIGUOUS"] or img.shape != (self.H, self.W):
            raise ValueError("img must be a C-contiguous float32 array of shape (%d, %d)" % (self.H, self.W))
        r = Result()
        self._ck(self._L.lfd_run_pass(self.h, pass_, img.ctypes.data_as(ctypes.c_void_p), flags, 1 if writeback else 0,
                                      ctypes.byref(r)))
        self._n = 1
        return r

    def blot(self, img, rects):
        rects = np.ascontiguousarray(rects, np.int32).reshape(-1, 4)
        self._ck(self._L.lfd_blot(self.h, img.ctypes.data_as(ctypes.c_void_p), rects.ctypes.data_as(ctypes.c_void_p), len(rects)))
        return img

    def stage_count(self, frame, pass_, stage):
        c = ctypes.c_int()
        self._ck(self._L.lfd_get_stage_count(self.h, frame, pass_, STAGES[stage], ctypes.byref(c)))
        return c.value

    def stage(self, frame, pass_, stage):
        sid = STAGES[stage]
        H, W = self.H, self.W
        if stage in ("mask", "gray", "equ", "eroded", "morph", "canny", "box", "nms"):
            out = np.empty((H, W), np.uint8)
        elif stage == "hist":
            out = np.empty(256, np.uint32)
        elif stage == "lut":
            out = np.empty(256, np.uint8)
        elif stage in ("fg_labels", "bg_labels"):
            out = np.empty((H, W), np.int32)
        elif stage in ("clipped", "input"):
            out = np.empty((H, W), np.float32)
        elif stage == "rects":
            out = np.zeros(self.stage_count(frame, pass_, stage), RECT_DTYPE)
        elif stage == "rect_screen":
            out = np.zeros(self.stage_count(frame, pass_, stage), np.int32)
        elif stage in ("accum_equ", "accum_box"):
            out = np.empty(self.stage_count(frame, pass_, stage), np.int32)
        elif stage in ("lines_equ", "lines_box"):
            out = np.empty((max(self.stage_count(frame, pass_, stage), 0), 1, 2), np.float32)
        else:
            raise KeyError(stage)
        if out.size:
            self._ck(self._L.lfd_get_stage(self.h, frame, pass_, sid, out.ctypes.data_as(ctypes.c_void_p), out.nbytes))
        return out

    def hough_lines(self, img, rho, theta, threshold, want_accum=False, max_lines=None):
        """cv2.HoughLines(img, rho, theta, threshold) -> (lines (n,1,2) float32 | None, accum | None)."""
        img = np.ascontiguousarray(img, np.uint8)
        Hh, Ww = img.shape
        na, nr = ctypes.c_int(), ctypes.c_int()
        self._L.lfd_hough_dims(Hh, Ww, float(rho), float(theta), ctypes.byref(na), ctypes.byref(nr))
        cap = na.value * nr.value if max_lines is None else max_lines       # max_lines=0: count + accumulator only, no sort
        lines = np.empty((max(cap, 1), 2), np.float32)
        accum = np.empty((na.value + 2, nr.value + 2), np.int32) if want_accum else None
        n = ctypes.c_int()
        self._ck(self._L.lfd_hough_lines(self.h, img.ctypes.data_as(ctypes.c_void_p), Hh, Ww, float(rho), float(theta),
                                         int(threshold), lines.ctypes.data_as(ctypes.c_void_p) if cap else None, cap, ctypes.byref(n),
                                         accum.ctypes.data_as(ctypes.c_void_p) if want_accum else None))
        k = min(n.value, cap)
        self.last_n_lines = n.value
        return (lines[:k].reshape(k, 1, 2).copy() if k else None), accum

    def canny(self, img, low, high):
        """cv2.Canny(img, low, high) for a uint8 image of this handle's frame size."""
        img = np.ascontiguousarray(img, np.uint8)
        if img.shape != (self.H, self.W):
            raise ValueError("image shape must be (%d, %d)" % (self.H, self.W))
        out = np.empty((self.H, self.W), np.uint8)
        self._ck(self._L.lfd_canny(self.h, img.ctypes.data_as(ctypes.c_void_p), int(low), int(high), out.ctypes.data_as(ctypes.c_void_p)))
        return out

    def smem_atomic_peak(self):
        """Measured peak shared-memory atomicAdd rate of the device, G atomics / s."""
        g = ctypes.c_double()
        self._ck(self._L.lfd_smem_atomic_peak(self.h, ctypes.byref(g)))
        return float(g.value)

    def fit_min_area_rect(self, img, contoursMode, contoursMethod, minAreaRectMinLen, lwTresh):
        """(detection, box_img) of processfield.py:201-263 for a uint8 image of this handle's frame size."""
        img = np.ascontiguousarray(img, np.uint8)
        if img.shape != (self.H, self.W):
            raise ValueError("image shape must be (%d, %d)" % (self.H, self.W))
        out = np.empty((self.H, self.W), np.uint8)
        det = ctypes.c_int()
        self._ck(self._L.lfd_fit_min_area_rect(self.h, img.ctypes.data_as(ctypes.c_void_p), int(contoursMode), int(contoursMethod),
                                               float(minAreaRectMinLen), float(lwTresh), out.ctypes.data_as(ctypes.c_void_p),
                                               ctypes.byref(det)))
        return bool(det.value), out

    def timings(self):
        ms = (ctypes.c_float * 32)()
        n = ctypes.c_int()
        self._ck(self._L.lfd_get_timings(self.h, ms, 32, ctypes.byref(n)))
        return [(self._L.lfd_timing_name(i).decode(), float(ms[i])) for i in range(n.value)]

    def kernel_times(self):
        """[(kernel name, pass, ms summed over the batch parts, launches)] of the bracketed kernels of the last batch."""
        out = []
        i = 0
        while True:
            name, p, ms, n = ctypes.c_char_p(), ctypes.c_int(), ctypes.c_float(), ctypes.c_int()
            if self._L.lfd_get_kernel_times(self.h, i, ctypes.byref(name), ctypes.byref(p), ctypes.byref(ms), ctypes.byref(n)) != LFD_OK:
                break
            if n.value:
                out.append((name.value.decode(), p.value, float(ms.value), n.value))
            i += 1
        return out

    def counters(self):
        c = (ctypes.c_int64 * 16)()
        self._ck(self._L.lfd_get_counters(self.h, c, 16))
        names = ["nnz_equ", "nnz_box", "votes", "runs_fg", "runs_bg", "contours", "passing_rects", "frames_dim",
                 "frames_hough", "frames_bright_run", "frames_dim_run", "rects_warp_path", "rects_thread_overflow",
                 "hough_smem_atomics", "ccl_lookback_stalls", "rects_screened"]
        return {k: int(c[i]) for i, k in enumerate(names)}

    def timer_mark(self, slot):
        """Record a CUDA event on this handle's stream (device-side benchmark timing)."""
        self._ck(self._L.lfd_timer_mark(self.h, slot))

    def timer_elapsed_ms(self, slot_start, end_handle=None, slot_end=1):
        ms = ctypes.c_float()
        eh = self if end_handle is None else end_handle
        self._ck(self._L.lfd_timer_elapsed(self.h, slot_start, eh.h, slot_end, ctypes.byref(ms)))
        return float(ms.value)

    def ktimings(self):
        """[(source line, ms)] per launch of the last run (only with LFD_KTIMING=1)."""
        lines = (ctypes.c_int * 1024)()
        ms = (ctypes.c_float * 1024)()
        n = ctypes.c_int()
        self._ck(self._L.lfd_get_ktimings(self.h, lines, ms, 1024, ctypes.byref(n)))
        return [(int(lines[i]), float(ms[i])) for i in range(n.value)]

    def kernel_launches(self):
        return int(self._L.lfd_kernel_launches(self.h))


_default = {}


def default_handle(height, width, device=0):
    """Process-wide single-frame handle used by the drop-in functions (one per frame shape and device)."""
    key = (height, width, device)
    h = _default.get(key)
    if h is None:
        h = Handle(height, width, max_batch=1, device=device)
        _default[key] = h
    return h
