"""ctypes loader for the CPU oracle (TEST INFRASTRUCTURE ONLY).

Only tests/, bench.py's cpu_baseline / ``--impl reference`` legs and
``__graft_entry__.smoke()`` may import this module.  The product package
``imageflow_b200`` never does (tests/test_boundary.py checks that).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libifb_oracle.so")

ERR_NAMES = {
    0: "OK", 1: "InvalidArgument", 2: "MethodNotImplemented", 3: "InvalidState",
    10: "TotalWeightZero", 11: "SourcePixelCountTooLarge", 12: "NoPixelInputs",
    13: "BadFilter", 14: "Capacity",
}
LOBE_NATURAL, LOBE_EXACT, LOBE_SHARPEN_PERCENT = 0, 1, 2
REPLACE_SELF, BLEND_WITH_SELF, BLEND_WITH_MATTE = 0, 1, 2


class Desc(C.Structure):
    """Binary-identical to ifb200_resample_desc (include/ifb200.h)."""
    _fields_ = [
        ("in_", C.c_void_p), ("in_w", C.c_uint32), ("in_h", C.c_uint32), ("in_stride", C.c_uint32),
        ("canvas", C.c_void_p), ("cv_w", C.c_uint32), ("cv_h", C.c_uint32), ("cv_stride", C.c_uint32),
        ("x", C.c_uint32), ("y", C.c_uint32), ("w", C.c_uint32), ("h", C.c_uint32),
        ("filter", C.c_int32), ("sharpen_percent", C.c_float), ("linear", C.c_int32),
        ("alpha_meaningful", C.c_int32), ("compose", C.c_int32), ("matte_bgra", C.c_uint8 * 4),
        ("color_matrix", C.c_void_p),
    ]


def build(force: bool = False) -> str:
    """Compile oracle/ifb_oracle.c with the committed Makefile (gcc only)."""
    src = os.path.join(_HERE, "ifb_oracle.c")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s", "CC=gcc"], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    return _LIB_PATH


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        build()
    L = C.CDLL(_LIB_PATH)
    u32p, f32p, u8p = C.POINTER(C.c_uint32), C.POINTER(C.c_float), C.POINTER(C.c_uint8)
    L.ifo_weights.argtypes = [C.c_int, C.c_double, C.c_int, C.c_float, C.c_uint32, C.c_uint32, u32p, u32p, u32p, f32p, C.c_size_t]
    L.ifo_weights.restype = C.c_int
    L.ifo_percent_negative_weight.argtypes = [C.c_int, C.c_double]
    L.ifo_percent_negative_weight.restype = C.c_double
    L.ifo_filter_eval.argtypes = [C.c_int, C.c_double, C.c_double]
    L.ifo_filter_eval.restype = C.c_double
    L.ifo_byte_to_float_table.argtypes = [C.c_int, f32p]
    L.ifo_linear_to_srgb_table.argtypes = [u8p]
    L.ifo_floatspace_to_srgb.argtypes = [C.c_int, C.c_float]
    L.ifo_floatspace_to_srgb.restype = C.c_uint8
    L.ifo_uchar_clamp_ff.argtypes = [C.c_float]
    L.ifo_uchar_clamp_ff.restype = C.c_uint8
    L.ifo_scale_and_render.argtypes = [C.POINTER(Desc)]
    L.ifo_scale_and_render.restype = C.c_int
    L.ifo_scale_and_render_batch.argtypes = [C.POINTER(Desc), C.c_size_t, C.c_int]
    L.ifo_scale_and_render_batch.restype = C.c_int
    L.ifo_resample_stages.argtypes = [C.POINTER(Desc), f32p, f32p]
    L.ifo_resample_stages.restype = C.c_int
    L.ifo_color_matrix.argtypes = [u8p, C.c_uint32, C.c_uint32, C.c_uint32, f32p]
    L.ifo_color_filter_matrix.argtypes = [C.c_int, C.c_float, f32p]
    L.ifo_color_filter_matrix.restype = C.c_int
    L.ifo_apply_matte.argtypes = [u8p, C.c_uint32, C.c_uint32, C.c_uint32, u8p, C.c_int]
    L.ifo_transpose.argtypes = [u8p, C.c_uint32, C.c_uint32, C.c_uint32, u8p, C.c_uint32]
    L.ifo_flip_vertical.argtypes = [u8p, C.c_uint32, C.c_uint32, C.c_uint32]
    L.ifo_flip_horizontal.argtypes = [u8p, C.c_uint32, C.c_uint32, C.c_uint32]
    L.ifo_white_balance.argtypes = [u8p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_float, u8p]
    L.ifo_max_threads.restype = C.c_int
    _lib = L
    return L


class OracleError(RuntimeError):
    def __init__(self, code: int):
        super().__init__(f"oracle error {code} ({ERR_NAMES.get(code, '?')})")
        self.code = code


def weights(filter_id: int, out_size: int, in_size: int, kernel_width_scale: float = 1.0,
            lobe_mode: int = LOBE_NATURAL, lobe_value: float = 0.0):
    """-> list of (left, right, np.float32 weights) per output sample; raises OracleError."""
    L = lib()
    left = np.zeros(out_size, np.uint32)
    right = np.zeros(out_size, np.uint32)
    off = np.zeros(out_size + 1, np.uint32)
    cap = out_size * (int(2 * (6.5 * max(1.0, in_size / max(out_size, 1)) * max(kernel_width_scale, 1.0))) + 8)
    w = np.zeros(cap, np.float32)
    rc = L.ifo_weights(filter_id, kernel_width_scale, lobe_mode, lobe_value, out_size, in_size,
                       left.ctypes.data_as(C.POINTER(C.c_uint32)), right.ctypes.data_as(C.POINTER(C.c_uint32)),
                       off.ctypes.data_as(C.POINTER(C.c_uint32)), w.ctypes.data_as(C.POINTER(C.c_float)), cap)
    if rc:
        raise OracleError(rc)
    return [(int(left[i]), int(right[i]), w[off[i]:off[i + 1]].copy()) for i in range(out_size)]


def byte_to_float_table(linear: bool) -> np.ndarray:
    t = np.zeros(256, np.float32)
    lib().ifo_byte_to_float_table(int(linear), t.ctypes.data_as(C.POINTER(C.c_float)))
    return t


def linear_to_srgb_table() -> np.ndarray:
    t = np.zeros(16384, np.uint8)
    lib().ifo_linear_to_srgb_table(t.ctypes.data_as(C.POINTER(C.c_uint8)))
    return t


def make_desc(inp: np.ndarray, canvas: np.ndarray, *, x=0, y=0, w=None, h=None, filter=2, sharpen=0.0,
              linear=True, alpha_meaningful=False, compose=REPLACE_SELF, matte=(0, 0, 0, 0), color_matrix=None,
              keep=None) -> Desc:
    """inp/canvas: C-contiguous-rows uint8 arrays of shape (H, stride_bytes//4 or W, 4) or (H, stride_bytes)."""
    def geom(a):
        assert a.dtype == np.uint8 and a.strides[-1] == 1
        hh = a.shape[0]
        stride = a.strides[0]
        ww = a.shape[1] if a.ndim == 3 else a.shape[1] // 4
        return hh, ww, stride
    ih, iw, istr = geom(inp)
    ch, cw, cstr = geom(canvas)
    d = Desc()
    d.in_ = inp.ctypes.data; d.in_w, d.in_h, d.in_stride = iw, ih, istr
    d.canvas = canvas.ctypes.data; d.cv_w, d.cv_h, d.cv_stride = cw, ch, cstr
    d.x, d.y = x, y
    d.w = cw - x if w is None else w
    d.h = ch - y if h is None else h
    d.filter = int(filter); d.sharpen_percent = float(sharpen); d.linear = int(bool(linear))
    d.alpha_meaningful = int(bool(alpha_meaningful)); d.compose = int(compose)
    d.matte_bgra = (C.c_uint8 * 4)(*matte)
    if color_matrix is not None:
        cm = np.ascontiguousarray(color_matrix, np.float32).reshape(25)
        d.color_matrix = cm.ctypes.data
        if keep is not None:
            keep.append(cm)
        else:
            d._cm = cm
    else:
        d.color_matrix = None
    d._refs = (inp, canvas)
    return d


def scale_and_render(inp: np.ndarray, canvas: np.ndarray, **kw) -> None:
    d = make_desc(inp, canvas, **kw)
    rc = lib().ifo_scale_and_render(C.byref(d))
    if rc:
        raise OracleError(rc)


def resample_stages(inp: np.ndarray, canvas: np.ndarray, **kw):
    d = make_desc(inp, canvas, **kw)
    v = np.zeros((d.in_h, d.w, 4), np.float32)
    hh = np.zeros((d.h, d.w, 4), np.float32)
    rc = lib().ifo_resample_stages(C.byref(d), v.ctypes.data_as(C.POINTER(C.c_float)), hh.ctypes.data_as(C.POINTER(C.c_float)))
    if rc:
        raise OracleError(rc)
    return v, hh


def synth_noise(w: int, h: int, seed: int = 0, alpha_mode: str = "opaque") -> np.ndarray:
    """imageflow_b200.synth.noise_np, generated by the C library (same bytes, ~100x faster)"""
    a = np.empty((h, w, 4), np.uint8)
    L = lib()
    L.ifo_synth_noise.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int]
    L.ifo_synth_noise.restype = None
    L.ifo_synth_noise(a.ctypes.data, w, h, a.strides[0], seed & 0xFFFFFFFF, int(alpha_mode != "opaque"))
    return a


def color_matrix(px: np.ndarray, m) -> None:
    m = np.ascontiguousarray(m, np.float32).reshape(25)
    h, w = px.shape[0], px.shape[1]
    lib().ifo_color_matrix(px.ctypes.data_as(C.POINTER(C.c_uint8)), w, h, px.strides[0], m.ctypes.data_as(C.POINTER(C.c_float)))


def color_filter_matrix(which: int, p: float = 0.0) -> np.ndarray:
    m = np.zeros(25, np.float32)
    rc = lib().ifo_color_filter_matrix(which, p, m.ctypes.data_as(C.POINTER(C.c_float)))
    if rc:
        raise OracleError(rc)
    return m.reshape(5, 5)


def apply_matte(px: np.ndarray, matte_bgra, alpha_meaningful=True) -> None:
    mm = (C.c_uint8 * 4)(*matte_bgra)
    lib().ifo_apply_matte(px.ctypes.data_as(C.POINTER(C.c_uint8)), px.shape[1], px.shape[0], px.strides[0], mm, int(alpha_meaningful))


def transpose(src: np.ndarray, dst: np.ndarray) -> None:
    """src (H, Ws, 4), dst (W, Hs, 4) uint8 with padded row strides allowed; dst[x, y] = src[y, x] for x < w, y < h."""
    u8p = C.POINTER(C.c_uint8)
    h, w = src.shape[0], dst.shape[0]
    lib().ifo_transpose(src.ctypes.data_as(u8p), src.strides[0], w, h, dst.ctypes.data_as(u8p), dst.strides[0])


def flip_vertical(px: np.ndarray, w=None) -> None:
    lib().ifo_flip_vertical(px.ctypes.data_as(C.POINTER(C.c_uint8)), px.shape[1] if w is None else w, px.shape[0], px.strides[0])


def flip_horizontal(px: np.ndarray, w=None) -> None:
    lib().ifo_flip_horizontal(px.ctypes.data_as(C.POINTER(C.c_uint8)), px.shape[1] if w is None else w, px.shape[0], px.strides[0])


def white_balance(px: np.ndarray, threshold=None, w=None) -> np.ndarray:
    """in place; returns the (3, 256) byte maps (R, G, B)."""
    maps = np.zeros((3, 256), np.uint8)
    u8p = C.POINTER(C.c_uint8)
    lib().ifo_white_balance(px.ctypes.data_as(u8p), px.shape[1] if w is None else w, px.shape[0], px.strides[0],
                            -1.0 if threshold is None else float(threshold), maps.ctypes.data_as(u8p))
    return maps


def detect_content(px: np.ndarray, threshold: int = 1, alpha_meaningful: bool = True, w=None):
    """graphics/whitespace.rs:284-331 -> ((x1, y1, x2, y2), number of window-interior pixels evaluated)."""
    L = lib()
    L.ifo_detect_content.argtypes = [C.POINTER(C.c_uint8), C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_uint32,
                                     C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)]
    L.ifo_detect_content.restype = C.c_int
    rect = (C.c_uint32 * 4)(); n = C.c_uint64()
    rc = L.ifo_detect_content(px.ctypes.data_as(C.POINTER(C.c_uint8)), px.shape[1] if w is None else w, px.shape[0], px.strides[0],
                              int(alpha_meaningful), int(threshold), rect, C.byref(n))
    if rc:
        raise OracleError(rc)
    return tuple(rect), n.value


def whitespace_codes(px: np.ndarray, threshold: int = 1, alpha_meaningful: bool = True) -> np.ndarray:
    """per-pixel code of sobel_scharr_detect (see ifb_oracle.h), shape (h, w) uint8."""
    L = lib()
    L.ifo_whitespace_codes.argtypes = [C.POINTER(C.c_uint8), C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_uint32, C.POINTER(C.c_uint8)]
    L.ifo_whitespace_codes.restype = None
    h, w = px.shape[0], px.shape[1]
    m = np.zeros((h, w), np.uint8)
    L.ifo_whitespace_codes(px.ctypes.data_as(C.POINTER(C.c_uint8)), w, h, px.strides[0], int(alpha_meaningful), int(threshold),
                           m.ctypes.data_as(C.POINTER(C.c_uint8)))
    return m


def detect_content_from_codes(codes: np.ndarray):
    """the window walk of detect_content replayed over a code map (whitespace_codes) -> ((x1, y1, x2, y2), centres)."""
    L = lib()
    L.ifo_detect_content_from_codes.argtypes = [C.POINTER(C.c_uint8), C.c_uint32, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)]
    L.ifo_detect_content_from_codes.restype = C.c_int
    codes = np.ascontiguousarray(codes, np.uint8)
    rect = (C.c_uint32 * 4)(); n = C.c_uint64()
    rc = L.ifo_detect_content_from_codes(codes.ctypes.data_as(C.POINTER(C.c_uint8)), codes.shape[1], codes.shape[0], rect, C.byref(n))
    if rc:
        raise OracleError(rc)
    return tuple(rect), n.value


# ---------------------------------------------------------------------------------------------- oracle/_ref: the reference itself
_REF_IDCT = os.path.join(_HERE, "_ref", "libidct_ref.so")


def idct_ref_available() -> bool:
    """oracle/_ref/libidct_ref.so = the reference's c_components/lib/codecs_jpeg_idct_fast.c compiled as it is (oracle/Makefile,
    run by __graft_entry__.build() where the reference tree is readable)."""
    return os.path.exists(_REF_IDCT)


_idct = None


def flow_scale_spatial_ref(samples: np.ndarray, n: int, srgb: bool = False) -> np.ndarray:
    """The reference's own flow_scale_spatial[_srgb]_{n}x{n} called block by block over a plane (H x W uint8, multiples of 8)."""
    global _idct
    if _idct is None:
        _idct = C.CDLL(_REF_IDCT)
    fn = getattr(_idct, f"flow_scale_spatial_{'srgb_' if srgb else ''}{n}x{n}")
    fn.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
    fn.restype = None
    a = np.ascontiguousarray(samples, np.uint8)
    h, w = a.shape
    out = np.zeros((h // 8 * n, w // 8 * n), np.uint8)
    rows = (C.c_void_p * n)()
    blk = np.zeros(64, np.uint8)
    for by in range(h // 8):
        for r in range(n):
            rows[r] = out.ctypes.data + (by * n + r) * out.strides[0]
        for bx in range(w // 8):
            blk[:] = a[by * 8:by * 8 + 8, bx * 8:bx * 8 + 8].reshape(64)
            fn(blk.ctypes.data, rows, bx * n)
    return out
