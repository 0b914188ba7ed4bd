"""
oracle.py — Python face of the two CPU checkers. TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module. The product (ngx_http_imgproc_b200/) never does.

  * `orc.*` / `run_chain()`  — the C restatement (oracle/imp_oracle.c) plus a restatement of the
    reference's argument grammar and stage order (bridge.c:18-281, 574-656; filters.c:43-455).
  * `Ref`                    — the reference's own filters.c/helpers.c/bridge.c compiled unmodified
    (oracle/_ref/libimp_ref.so, built by oracle/Makefile when /root/reference is present), driven
    either op-by-op through IplImage headers or end to end through RunJob with a RAW codec.
    OpenCV calls inside it go to cv2 (4.13, IPP off) when `Ref.use_cv2()` was called and cv2 is
    importable, else to the C restatement.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from dataclasses import dataclass, field
from typing import List, Optional, Tuple

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

IMP_OK = 0
IMP_ERROR_INVALID_ARGS = 50
IMP_ERROR_NO_SUCH_FILTER = 52
IMP_ERROR_NO_SUCH_WATERMARK = 53
IMP_ERROR_TOO_BIG_TARGET = 54
IMP_ERROR_TOO_MUCH_FILTERS = 55
STEP_START, STEP_VALIDATE, STEP_DECODE, STEP_CROP, STEP_RESIZE, STEP_FILTERING, STEP_WATERMARK, STEP_INFO, STEP_ENCODE = range(9)

NN, LINEAR, CUBIC, AREA = 0, 1, 2, 3


def build(force: bool = False) -> None:
    """make -C oracle (the restatement always; _ref only when /root/reference exists)."""
    so = os.path.join(HERE, "libimp_oracle.so")
    if force or not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(os.path.join(HERE, "imp_oracle.c")) \
            or (os.path.isdir("/root/reference") and not os.path.exists(os.path.join(HERE, "_ref", "libimp_ref.so"))):
        subprocess.run(["make", "-C", HERE], check=True, stdout=subprocess.DEVNULL)


class _Img(C.Structure):
    _fields_ = [("data", C.c_void_p), ("width", C.c_int), ("height", C.c_int), ("channels", C.c_int), ("step", C.c_int)]


def _view(a: np.ndarray) -> _Img:
    assert a.dtype == np.uint8 and a.ndim == 3 and a.strides[2] == 1 and a.strides[1] == a.shape[2]
    return _Img(a.ctypes.data, a.shape[1], a.shape[0], a.shape[2], a.strides[0])


def _as3(a: np.ndarray) -> np.ndarray:
    return a[:, :, None] if a.ndim == 2 else a


class _Orc:
    """ctypes bindings of oracle/imp_oracle.c. All functions take/return HxWxC uint8 arrays."""

    def __init__(self):
        build()
        self.lib = C.CDLL(os.path.join(HERE, "libimp_oracle.so"))
        L = self.lib
        L.orc_vignette_mask.restype = C.c_float
        L.orc_vignette_mask.argtypes = [C.c_int] * 4 + [C.c_float] * 2
        L.orc_vignette_mask_table.argtypes = [C.c_void_p] + [C.c_int] * 4 + [C.c_float] * 2
        L.orc_perceived_brightness.restype = C.c_float
        for n in ("orc_add_color",):
            getattr(L, n).argtypes = [C.c_void_p, C.c_void_p, C.c_float]
        L.orc_gamma.argtypes = [C.c_void_p, C.c_float]
        L.orc_gamma_lut.argtypes = [C.c_float, C.c_void_p]
        L.orc_brightness_contrast.argtypes = [C.c_void_p, C.c_float, C.c_float]
        L.orc_vignette.argtypes = [C.c_void_p, C.c_float, C.c_float]
        L.orc_scanline.argtypes = [C.c_void_p, C.c_float, C.c_float, C.c_int, C.c_int]
        L.orc_alpha_over.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_float]
        L.orc_gaussian.argtypes = [C.c_void_p, C.c_void_p, C.c_double]
        L.orc_gaussian_taps.argtypes = [C.c_double, C.c_void_p, C.c_int]
        L.orc_watermark_origin.argtypes = [C.c_int] * 4 + [C.c_char, C.c_char, C.c_int, C.c_int, C.c_void_p, C.c_void_p]

    # -- in-place pixel ops (return a new array; input untouched) --------------------------------
    def _inplace(self, fn, img, *args):
        out = np.ascontiguousarray(img).copy()
        v = _view(out)
        getattr(self.lib, fn)(C.byref(v), *args)
        return out

    def rgb2hsv(self, img): return self._inplace("orc_rgb2hsv", img)
    def hsv2rgb(self, img): return self._inplace("orc_hsv2rgb", img)
    def modulate(self, img, h, s, v): return self._inplace("orc_modulate_hsv", img, (C.c_int * 3)(h, s, v))
    def add_color(self, img, rgb, alpha): return self._inplace("orc_add_color", img, (C.c_int * 3)(*rgb), C.c_float(alpha))
    def gamma(self, img, g): return self._inplace("orc_gamma", img, C.c_float(g))
    def contrast(self, img, br, ct): return self._inplace("orc_brightness_contrast", img, C.c_float(br), C.c_float(ct))
    def vignette(self, img, intensity, radius=1.0): return self._inplace("orc_vignette", img, C.c_float(intensity), C.c_float(radius))
    def lomo(self, img): return self._inplace("orc_lomo", img)
    def gotham(self, img): return self._inplace("orc_gotham", img)
    def kelvin(self, img): return self._inplace("orc_kelvin", img)
    def rainbow(self, img, sat): return self._inplace("orc_rainbow", img, C.c_int(sat))
    def scanline(self, img, intensity, opacity, freq, width):
        return self._inplace("orc_scanline", img, C.c_float(intensity), C.c_float(opacity), C.c_int(freq), C.c_int(width))
    def paper(self, img): return self._inplace("orc_blend_with_paper", img)

    def gamma_lut(self, g):
        lut = (C.c_int * 256)()
        self.lib.orc_gamma_lut(C.c_float(g), lut)
        return np.array(lut, dtype=np.int64)

    def gradient_lut(self, colors: np.ndarray):
        colors = np.ascontiguousarray(colors, dtype=np.uint8)
        lut = np.zeros(768, np.uint8)
        self.lib.orc_gradient_lut(C.c_void_p(colors.ctypes.data), C.c_int(len(colors)), C.c_void_p(lut.ctypes.data))
        return lut

    def gradmap(self, img, colors):
        lut = self.gradient_lut(np.asarray(colors, np.uint8).reshape(-1, 3))
        return self._inplace("orc_gradmap", img, C.c_void_p(lut.ctypes.data))

    def alpha_over(self, dst, x0, y0, src, opacity):
        out = np.ascontiguousarray(dst).copy()
        s = np.ascontiguousarray(src)
        dv, sv = _view(out), _view(s)
        self.lib.orc_alpha_over(C.byref(dv), x0, y0, C.byref(sv), C.c_float(opacity))
        return out

    def watermark_origin(self, bw, bh, ow, oh, gx, gy, ox, oy):
        x0, y0 = C.c_int(0), C.c_int(0)
        ok = self.lib.orc_watermark_origin(bw, bh, ow, oh, gx.encode(), gy.encode(), ox, oy, C.byref(x0), C.byref(y0))
        return (x0.value, y0.value) if ok else None

    def perceived_brightness(self, img):
        v = _view(np.ascontiguousarray(img))
        return float(self.lib.orc_perceived_brightness(C.byref(v)))

    def gif_expand(self, frames, cw, ch, destructive):
        """frames: list of dicts(indices HxW uint8 bottom-up (or H x pitch with `width` given: the page block as FreeImage
        pads it), left, top, dispose, key, palette 256x4). Returns n BGRA canvases."""
        class F(C.Structure):
            _fields_ = [("indices", C.c_void_p), ("pitch", C.c_int), ("width", C.c_int), ("height", C.c_int), ("left", C.c_int),
                        ("top", C.c_int), ("dispose", C.c_int), ("key", C.c_int), ("palette", C.c_void_p)]
        keep, arr = [], (F * len(frames))()
        for i, f in enumerate(frames):
            idx = np.ascontiguousarray(f["indices"], np.uint8); pal = np.ascontiguousarray(f["palette"], np.uint8)
            keep += [idx, pal]
            arr[i] = F(idx.ctypes.data, idx.strides[0], f.get("width") or idx.shape[1], idx.shape[0], f["left"], f["top"], f["dispose"], f["key"], pal.ctypes.data)
        outs = [np.zeros((ch, cw, 4), np.uint8) for _ in frames]
        ptrs = (C.c_void_p * len(frames))(*[o.ctypes.data for o in outs])
        self.lib.orc_gif_expand(arr, len(frames), cw, ch, 1 if destructive else 0, ptrs, cw * 4)
        return outs

    def ascii(self, img, wide=False) -> bytes:
        a = np.ascontiguousarray(img)
        v = _view(a)
        n = (a.shape[1] + 1) * a.shape[0] - 1
        out = C.create_string_buffer(n + 1)
        self.lib.orc_ascii.restype = C.c_long
        self.lib.orc_ascii(C.byref(v), 1 if wide else 0, out)
        return out.raw[:n]

    def vignette_mask(self, x, y, w, h, power, radius):
        return float(self.lib.orc_vignette_mask(x, y, w, h, C.c_float(power), C.c_float(radius)))

    def vignette_mask_table(self, nx, ny, w, h, power, radius):
        """vignette_mask at |dx| = i < nx, |dy| = j < ny from the frame's centre: float32 (ny, nx)."""
        out = np.empty((ny, nx), np.float32)
        self.lib.orc_vignette_mask_table(out.ctypes.data_as(C.c_void_p), nx, ny, w, h, C.c_float(power), C.c_float(radius))
        return out

    # -- geometry ------------------------------------------------------------------------------
    def crop(self, img, x, y, w, h):
        src = np.ascontiguousarray(img)
        out = np.empty((h, w, src.shape[2]), np.uint8)
        sv, dv = _view(src), _view(out)
        self.lib.orc_copy_roi(C.byref(sv), x, y, C.byref(dv))
        return out

    def resize(self, img, dw, dh, mode):
        src = np.ascontiguousarray(img)
        out = np.empty((dh, dw, src.shape[2]), np.uint8)
        sv, dv = _view(src), _view(out)
        self.lib.orc_resize(C.byref(sv), C.byref(dv), mode)
        return out

    def flip(self, img, mode):
        src = np.ascontiguousarray(img)
        out = np.empty_like(src)
        sv, dv = _view(src), _view(out)
        self.lib.orc_flip(C.byref(sv), C.byref(dv), mode)
        return out

    def transpose(self, img):
        src = np.ascontiguousarray(img)
        out = np.empty((src.shape[1], src.shape[0], src.shape[2]), np.uint8)
        sv, dv = _view(src), _view(out)
        self.lib.orc_transpose(C.byref(sv), C.byref(dv))
        return out

    def gray2bgr(self, img):
        src = np.ascontiguousarray(_as3(img))
        out = np.empty((src.shape[0], src.shape[1], 3), np.uint8)
        sv, dv = _view(src), _view(out)
        self.lib.orc_gray2bgr(C.byref(sv), C.byref(dv))
        return out

    def gaussian(self, img, sigma):
        src = np.ascontiguousarray(img)
        out = np.empty_like(src)
        sv, dv = _view(src), _view(out)
        self.lib.orc_gaussian(C.byref(sv), C.byref(dv), C.c_double(float(np.float32(sigma))))
        return out

    def gaussian_taps(self, sigma):
        buf = (C.c_int * 4096)()
        n = self.lib.orc_gaussian_taps(C.c_double(sigma), buf, 4096)
        return list(buf[:n])


_orc: Optional[_Orc] = None


def orc() -> _Orc:
    global _orc
    if _orc is None:
        _orc = _Orc()
    return _orc


# ------------------------------------------------------------------------------------------------
# Restatement of the reference's argument grammar + stage order (Python; strtol/strtof via libc)
# ------------------------------------------------------------------------------------------------
_libc = C.CDLL(None)
_libc.strtol.restype = C.c_long
_libc.strtol.argtypes = [C.c_char_p, C.POINTER(C.c_char_p), C.c_int]
_libc.strtof.restype = C.c_float
_libc.strtof.argtypes = [C.c_char_p, C.POINTER(C.c_char_p)]


def c_strtol(s: str, base: int = 10) -> Tuple[int, str]:
    b = s.encode("latin-1")
    buf = C.create_string_buffer(b)
    end = C.c_char_p()
    v = _libc.strtol(buf, C.byref(end), base)
    consumed = C.cast(end, C.c_void_p).value - C.addressof(buf)
    return int(v), b[consumed:].decode("latin-1")


def c_strtof(s: str) -> float:
    return float(_libc.strtof(s.encode("latin-1"), None))


def _tokens(s: str, sep: str = ",") -> List[str]:
    """strtok_r semantics: runs of separators collapse, no empty tokens."""
    return [t for t in s.split(sep) if t != ""]


def _u32(v: int) -> int:
    return v & 0xFFFFFFFF


def _i32(v: int) -> int:
    v &= 0xFFFFFFFF
    return v - (1 << 32) if v & 0x80000000 else v


def _round_half_away(x: float) -> int:
    import math
    return int(math.floor(x + 0.5)) if x >= 0 else int(math.ceil(x - 0.5))


@dataclass
class OracleConfig:
    """Mirror of the Config fields the hot path reads (required.h:110-120)."""
    max_w: int = 2000                 # MaxTargetDimensions (module.c:117-190 defaults)
    max_h: int = 2000
    max_filters: int = 5
    allow_experiments: bool = False
    watermark: Optional[np.ndarray] = None      # decoded overlay HxWx{3,4}
    wm_gravity_x: str = "l"
    wm_gravity_y: str = "t"
    wm_offset_x: int = 0
    wm_offset_y: int = 0
    wm_opacity: int = 100


def parse_crop(args: str, gravity: Optional[str], col: int, row: int):
    """bridge.c:18-128. Returns (code, (x, y, w, h))."""
    f32 = np.float32
    toks = _tokens(args)
    ww, wwmode = c_strtol(toks[0] if len(toks) > 0 else "")
    wh, whmode = c_strtol(toks[1] if len(toks) > 1 else "")
    ww, wh = _u32(ww), _u32(wh)
    rest = toks[2:]
    respect = False
    if gravity is not None:
        if len(gravity) > 2:
            respect = True
        else:
            return IMP_ERROR_INVALID_ARGS, None
    if wwmode == "" and whmode == "":
        with np.errstate(all="ignore"):
            px = f32(col)
            py = f32(f32(px / f32(ww)) * f32(wh))
            if py > f32(row):
                py = f32(row)
                px = f32(f32(py / f32(wh)) * f32(ww))
        # (int)round(px): NaN/inf -> INT_MIN on x86
        def cv(v):
            v = float(v)
            if v != v or abs(v) >= 2147483648.0:
                return _u32(-(1 << 31))
            return _u32(_round_half_away(v))
        ww, wh = cv(px), cv(py)
    elif wwmode == "px" and whmode == "px":
        pass
    else:
        return IMP_ERROR_INVALID_ARGS, None
    if ww == 0 or ww > col or wh == 0 or wh > row:
        return IMP_ERROR_INVALID_ARGS, None
    gtoks = _tokens(gravity) if respect else rest

    def axis(tok, lo_key, hi_key, size, win, default):
        if tok is None:
            tok = default
        if tok == lo_key:
            return 0
        if tok == hi_key:
            return size - win
        if tok == "c":
            return _round_half_away((size - win) / 2.0)
        v, mode = c_strtol(tok)
        if mode == "px":
            return _i32(_u32(v))
        return None

    tx = gtoks[0] if len(gtoks) > 0 else None
    ty = gtoks[1] if len(gtoks) > 1 else None
    if respect and (tx is None or ty is None):
        # the reference would strcmp(NULL): undefined; treat as invalid
        return IMP_ERROR_INVALID_ARGS, None
    x = axis(tx, "l", "r", col, ww, "c")
    if x is None:
        return IMP_ERROR_INVALID_ARGS, None
    y = axis(ty, "t", "b", row, wh, "t")
    if y is None:
        return IMP_ERROR_INVALID_ARGS, None
    if x + ww > col or y + wh > row:
        return IMP_ERROR_INVALID_ARGS, None
    if x < 0 or y < 0:
        return IMP_ERROR_INVALID_ARGS, None      # reference: cvCopy size-mismatch assert inside OpenCV
    return IMP_OK, (x, y, ww, wh)


def parse_resize(args: str, col: int, row: int, cfg: OracleConfig, simple: bool):
    """bridge.c:143-190. Returns (code, (w, h, mode))."""
    f32 = np.float32
    toks = _tokens(args)
    w = _u32(c_strtol(toks[0] if len(toks) > 0 else "")[0])
    h = _u32(c_strtol(toks[1] if len(toks) > 1 else "")[0])
    if w == 0 and h == 0:
        return IMP_ERROR_INVALID_ARGS, None
    if w == 0:
        w = _u32(_round_half_away(float(f32(f32(f32(h) / f32(row)) * f32(col)))))
    if h == 0:
        h = _u32(_round_half_away(float(f32(f32(f32(w) / f32(col)) * f32(row)))))
    up = len(toks) > 2 and toks[2] == "up"
    if not up:
        w = min(w, col)
        h = min(h, row)
    if (cfg.max_w > 0 and w > cfg.max_w) or (cfg.max_h > 0 and w > cfg.max_h):   # sic: width twice (bridge.c:184)
        return IMP_ERROR_TOO_BIG_TARGET, None
    if w == 0 or h == 0:
        return IMP_ERROR_INVALID_ARGS, None      # reference: cvCreateImage error inside OpenCV
    if w > 65535 or h > 65535:
        return IMP_ERROR_TOO_BIG_TARGET, None    # documented hard cap of the GPU path
    mode = NN if simple else (CUBIC if (w > col or h > row) else AREA)
    return IMP_OK, (w, h, mode)


EXPERIMENTAL = {"vignette", "gotham", "lomo", "kelvin", "rainbow", "scanline"}   # filters.c:19-24
FILTERS = ["flip", "rotate", "modulate", "colorize", "blur", "gamma", "contrast", "gradmap",
           "vignette", "gotham", "lomo", "kelvin", "rainbow", "scanline"]            # filters.c:10-24


def _hex3(tok: str) -> List[int]:
    return [c_strtol(tok[i * 2:i * 2 + 2], 16)[0] for i in range(3)]


def apply_filter(img: np.ndarray, request: str, allow_experiments: bool):
    """filters.c:43-70 Filter + the 14 callbacks (filters.c:72-455). Returns (code, image)."""
    o = orc()
    parts = _tokens(request, "=")
    if len(parts) == 0:
        return IMP_ERROR_NO_SUCH_FILTER, img
    if len(parts) < 2:
        return IMP_ERROR_INVALID_ARGS, img
    name, args = parts[0], parts[1]
    if name not in FILTERS or (name in EXPERIMENTAL and not allow_experiments):
        return IMP_ERROR_NO_SUCH_FILTER, img
    INV = IMP_ERROR_INVALID_ARGS
    if name == "flip":
        if len(args) != 2 or args[0] not in "01" or args[1] not in "01":
            return INV, img
        hz, vt = args[0] == "1", args[1] == "1"
        if hz and vt: return IMP_OK, o.flip(img, -1)
        if hz: return IMP_OK, o.flip(img, 1)
        if vt: return IMP_OK, o.flip(img, 0)
        return IMP_OK, img
    if name == "rotate":
        amount = _i32(c_strtol(args)[0])
        if amount in (90, 270):
            return IMP_OK, o.flip(o.transpose(img), 270 - amount)
        if amount == 180:
            return IMP_OK, o.flip(img, -1)
        return INV, img
    if name == "modulate":
        t = _tokens(args)
        if len(t) < 3: return INV, img
        p = [_i32(c_strtol(x)[0]) for x in t[:3]]
        if p[0] < 0 or p[0] > 180 or p[2] <= 0: return INV, img
        return IMP_OK, o.modulate(img, *p)
    if name == "colorize":
        t = _tokens(args)
        if len(t) == 0 or len(t[0]) != 6: return INV, img
        rgb = [_i32(v) for v in _hex3(t[0])]
        op = c_strtof(t[1]) if len(t) > 1 else 0.5
        if op < 0 or op > 1: return INV, img
        return IMP_OK, o.add_color(img, rgb, op)
    if name == "blur":
        t = _tokens(args)
        if len(t) == 0: return INV, img
        sigma = c_strtof(t[0])
        if sigma < 0: return INV, img
        if not sigma > 0: return INV, img        # sigma==0 / NaN: OpenCV asserts (App. C-9) -> INVALID_ARGS here
        return IMP_OK, o.gaussian(img, sigma)
    if name == "gamma":
        return IMP_OK, o.gamma(img, c_strtof(args))
    if name == "contrast":
        v = c_strtof(args)
        if not v > 0: return INV, img            # `value <= 0` is false for NaN in C; strtof never yields NaN from digits
        return IMP_OK, o.contrast(img, 0.0, v)
    if name == "gradmap":
        t = _tokens(args)
        if any(len(x) != 6 for x in t): return INV, img
        if len(t) < 2 or len(t) > 8: return INV, img   # reference: garbage LUT / heap overflow (App. C-4)
        cols = [[v & 0xFF for v in _hex3(x)] for x in t]
        return IMP_OK, o.gradmap(img, cols)
    if name == "vignette":
        t = _tokens(args)
        inten = c_strtof(t[0]) if len(t) > 0 else 0.5
        rad = c_strtof(t[1]) if len(t) > 1 else 1.0
        return IMP_OK, o.vignette(img, inten, rad)
    if name == "gotham": return IMP_OK, o.gotham(img)
    if name == "lomo": return IMP_OK, o.lomo(img)
    if name == "kelvin": return IMP_OK, o.kelvin(img)
    if name == "rainbow":
        sat = {"full": 255, "mid": 190, "pale": 120}.get(args)
        if sat is None: return INV, img
        return IMP_OK, o.rainbow(img, sat)
    if name == "scanline":
        t = _tokens(args)
        if len(t) == 0: return INV, img          # reference dereferences NULL (App. C-10)
        inten = c_strtof(t[0])
        if inten < 0 or inten > 1: return INV, img
        op = c_strtof(t[1]) if len(t) > 1 else 0.0
        if op < 0 or op > 1: return INV, img
        freq = _i32(c_strtol(t[2])[0]) if len(t) > 2 else 1
        if freq < 1: return INV, img
        width = _i32(c_strtol(t[3])[0]) if len(t) > 3 else 1
        if width < 1: return INV, img
        return IMP_OK, o.scanline(img, inten, op, freq, width)
    return IMP_ERROR_NO_SUCH_FILTER, img


def fi_pack(img: np.ndarray, bits: int) -> np.ndarray:
    """advancedio.c:65-101 IplToFI32 / IplToFI24: bottom-up rows; 32-bit gets alpha 255 when the frame has none,
    24-bit keeps the first three channels."""
    img = np.ascontiguousarray(img)[::-1]
    if bits == 32:
        if img.shape[2] == 4:
            return np.ascontiguousarray(img)
        out = np.full(img.shape[:2] + (4,), 255, np.uint8)
        out[:, :, :3] = img[:, :, :3]
        return out
    return np.ascontiguousarray(img[:, :, :3])


def run_chain(img: np.ndarray, crop: Optional[str] = None, gravity: Optional[str] = None,
              resize: Optional[str] = None, filters: Optional[List[str]] = None,
              cfg: Optional[OracleConfig] = None, simple: bool = False, flatten: bool = False,
              linear: bool = False, pack: int = 0):
    """RunJob steps 3-7 (bridge.c:574-656) on one decoded frame. Returns (code, step, image).
    `linear=True` is the shim-level INTER_LINEAR extension (not a reference call site)."""
    o = orc()
    cfg = cfg or OracleConfig()
    img = np.ascontiguousarray(_as3(img))
    step = STEP_CROP
    if crop is not None:
        code, win = parse_crop(crop, gravity, img.shape[1], img.shape[0])
        if code: return code, step, img
        img = o.crop(img, *win)
    step = STEP_RESIZE
    if resize is not None:
        code, r = parse_resize(resize, img.shape[1], img.shape[0], cfg, simple)
        if code: return code, step, img
        mode = r[2]
        if linear and mode != NN: mode = LINEAR
        img = o.resize(img, r[0], r[1], mode)
    step = STEP_FILTERING
    if img.shape[2] == 1:
        img = o.gray2bgr(img)
    for f in (filters or []):
        code, img = apply_filter(img, f, cfg.allow_experiments)
        if code: return code, step, img
    step = STEP_WATERMARK
    if cfg.watermark is not None:
        wm = np.ascontiguousarray(cfg.watermark)
        org = o.watermark_origin(img.shape[1], img.shape[0], wm.shape[1], wm.shape[0],
                                 cfg.wm_gravity_x, cfg.wm_gravity_y, cfg.wm_offset_x, cfg.wm_offset_y)
        if org is None:
            return IMP_ERROR_INVALID_ARGS, step, img      # reference aborts inside OpenCV (App. C-8)
        img = o.alpha_over(img, org[0], org[1], wm, float(np.float32(cfg.wm_opacity / 100.0)))
    if flatten and img.shape[2] == 4:
        img = o.paper(img)
    if pack:
        img = fi_pack(img, pack)
    return IMP_OK, STEP_ENCODE, img


def parse_query(query: str, cfg: OracleConfig):
    """bridge.c:346-372: '&'-separated tokens, prefix match in a fixed order, last one wins.
    Returns (code, dict)."""
    out = dict(crop=None, gravity=None, resize=None, quality=None, format=None, page=-1, filters=[])
    for tok in _tokens(query, "&"):
        def after(ch):
            i = tok.find(ch)
            return tok[i + 1:] if i >= 0 else None
        if tok.startswith("crop"): out["crop"] = after("=")
        elif tok.startswith("gravity"): out["gravity"] = after("=")
        elif tok.startswith("resize"): out["resize"] = after("=")
        elif tok.startswith("quality"): out["quality"] = after("=")
        elif tok.startswith("format"): out["format"] = after("=")
        elif tok.startswith("page"): out["page"] = c_strtol(after("=") or "")[0]
        elif tok.startswith("filter"):
            if len(out["filters"]) >= cfg.max_filters:
                return IMP_ERROR_TOO_MUCH_FILTERS, out
            out["filters"].append(after("-"))
    return IMP_OK, out


# ------------------------------------------------------------------------------------------------
# The compiled reference (oracle/_ref/libimp_ref.so)
# ------------------------------------------------------------------------------------------------
class IplROI(C.Structure):
    _fields_ = [("coi", C.c_int), ("xOffset", C.c_int), ("yOffset", C.c_int), ("width", C.c_int), ("height", C.c_int)]


class IplImage(C.Structure):
    pass


IplImage._fields_ = [
    ("nSize", C.c_int), ("ID", C.c_int), ("nChannels", C.c_int), ("alphaChannel", C.c_int), ("depth", C.c_int),
    ("colorModel", C.c_char * 4), ("channelSeq", C.c_char * 4),
    ("dataOrder", C.c_int), ("origin", C.c_int), ("align", C.c_int), ("width", C.c_int), ("height", C.c_int),
    ("roi", C.POINTER(IplROI)), ("maskROI", C.c_void_p), ("imageId", C.c_void_p), ("tileInfo", C.c_void_p),
    ("imageSize", C.c_int), ("imageData", C.c_void_p), ("widthStep", C.c_int),
    ("BorderMode", C.c_int * 4), ("BorderConst", C.c_int * 4), ("imageDataOrigin", C.c_void_p),
]


class _NgxStr(C.Structure):
    _fields_ = [("len", C.c_size_t), ("data", C.c_void_p)]


class _Position(C.Structure):
    _fields_ = [("GravityX", C.c_char), ("GravityY", C.c_char), ("OffsetX", C.c_int), ("OffsetY", C.c_int)]


class _Dimensions(C.Structure):
    _fields_ = [("W", C.c_uint), ("H", C.c_uint)]


class _CvSize(C.Structure):
    _fields_ = [("width", C.c_int), ("height", C.c_int)]


class _RecoverInfo(C.Structure):
    _fields_ = [("Size", _CvSize), ("Depth", C.c_int), ("Channels", C.c_int), ("Step", C.c_int),
                ("Length", C.c_size_t), ("Pointer", C.c_void_p)]


class _Config(C.Structure):
    _fields_ = [("Enable", C.c_ssize_t), ("MaxSrcSize", C.c_size_t), ("WatermarkPath", _NgxStr),
                ("WatermarkOpacity", C.c_ssize_t), ("WatermarkPosition", C.POINTER(_Position)),
                ("WatermarkInfo", C.POINTER(_RecoverInfo)), ("MaxTargetDimensions", C.POINTER(_Dimensions)),
                ("MaxFiltersCount", C.c_ssize_t), ("AllowExperiments", C.c_ssize_t)]


class Ref:
    """The reference's own C, compiled unmodified. `Ref.available()` is False on a box where neither
    /root/reference nor a prebuilt oracle/_ref/libimp_ref.so exists."""
    _lib = None
    _cbs = None

    @classmethod
    def path(cls):
        return os.path.join(HERE, "_ref", "libimp_ref.so")

    @classmethod
    def available(cls) -> bool:
        if cls._lib is not None:
            return True
        try:
            build()
        except Exception:
            pass
        return os.path.exists(cls.path())

    @classmethod
    def lib(cls):
        if cls._lib is None:
            if not cls.available():
                raise RuntimeError("oracle/_ref/libimp_ref.so not built (needs /root/reference)")
            cls._lib = C.CDLL(cls.path())
            L = cls._lib
            L.ref_sizeof_iplimage.restype = C.c_size_t
            L.ref_sizeof_config.restype = C.c_size_t
            assert L.ref_sizeof_iplimage() == C.sizeof(IplImage) == 144
            assert L.ref_sizeof_config() == C.sizeof(_Config)
            L.CalcPerceivedBrightness.restype = C.c_float
            L.AlphaBlendOver.argtypes = [C.c_void_p, C.c_void_p, C.c_float]
            L.cvCreateImage.restype = C.POINTER(IplImage)
            L.cvCreateImage.argtypes = [_CvSize, C.c_int, C.c_int]
            L.CalculateGammaLUT.restype = C.POINTER(C.c_int)
            L.CalculateGammaLUT.argtypes = [C.c_float]
            L.CalculateGradientLUT.restype = C.POINTER(C.c_ubyte)
        return cls._lib

    # -- cv2 backend for the OpenCV calls ------------------------------------------------------
    @classmethod
    def use_cv2(cls, enable: bool = True) -> bool:
        """Route cvResize/cvSmooth/cvFlip/cvTranspose inside the compiled reference to cv2 4.13
        (IPP off, 1 thread): the real OpenCV CPU path. Returns False if cv2 is missing."""
        L = cls.lib()
        if not enable:
            L.ref_set_callbacks.argtypes = [C.c_void_p] * 4
            L.ref_set_callbacks(None, None, None, None)
            cls._cbs = None
            return True
        try:
            import cv2
        except Exception:
            return False
        cv2.ipp.setUseIPP(False)
        cv2.setNumThreads(1)

        def arr(ptr, w, h, c, step):
            buf = (C.c_ubyte * (step * h)).from_address(ptr)
            a = np.frombuffer(buf, np.uint8).reshape(h, step)[:, :w * c].reshape(h, w, c)
            return a

        RES = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int)
        SMO = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double)
        FLP = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int)
        TRN = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int)

        def _res(s, sw, sh, sc, ss, d, dw, dh, ds, mode):
            out = cv2.resize(arr(s, sw, sh, sc, ss), (dw, dh), interpolation=mode)
            arr(d, dw, dh, sc, ds)[...] = out.reshape(dh, dw, sc)

        def _smo(s, w, h, c, st, sigma):
            a = arr(s, w, h, c, st)
            out = cv2.GaussianBlur(a, (0, 0), sigma, sigmaY=0, borderType=cv2.BORDER_REPLICATE)
            a[...] = out.reshape(h, w, c)

        def _flp(s, w, h, c, ss, d, ds, mode):
            arr(d, w, h, c, ds)[...] = cv2.flip(arr(s, w, h, c, ss), mode).reshape(h, w, c)

        def _trn(s, w, h, c, ss, d, ds):
            arr(d, h, w, c, ds)[...] = cv2.transpose(arr(s, w, h, c, ss)).reshape(w, h, c)

        cls._cbs = (RES(_res), SMO(_smo), FLP(_flp), TRN(_trn))
        L.ref_set_callbacks.argtypes = [RES, SMO, FLP, TRN]
        L.ref_set_callbacks(*cls._cbs)
        return True

    # -- IplImage helpers ------------------------------------------------------------------------
    @classmethod
    def new_image(cls, img: np.ndarray):
        """cvCreateImage + copy (so that the reference may cvReleaseImage it)."""
        L = cls.lib()
        img = _as3(img)
        h, w, c = img.shape
        p = L.cvCreateImage(_CvSize(w, h), 8, c)
        cls.to_numpy(p, writable=True)[...] = img
        return p

    @staticmethod
    def to_numpy(p, writable=False) -> np.ndarray:
        im = p.contents
        buf = (C.c_ubyte * (im.widthStep * im.height)).from_address(im.imageData)
        a = np.frombuffer(buf, np.uint8).reshape(im.height, im.widthStep)[:, :im.width * im.nChannels]
        a = a.reshape(im.height, im.width, im.nChannels)
        return a if writable else a.copy()

    @classmethod
    def release(cls, p):
        pp = C.POINTER(IplImage)(p.contents)
        cls.lib().cvReleaseImage(C.byref(pp))

    @classmethod
    def make_config(cls, cfg: OracleConfig):
        """Build a reference Config (required.h:110-120); returns (struct, keepalive)."""
        keep = []
        c = _Config()
        c.Enable = 1
        c.MaxSrcSize = 4 << 20
        c.WatermarkOpacity = cfg.wm_opacity
        pos = _Position(cfg.wm_gravity_x.encode(), cfg.wm_gravity_y.encode(), cfg.wm_offset_x, cfg.wm_offset_y)
        dims = _Dimensions(cfg.max_w, cfg.max_h)
        keep += [pos, dims]
        c.WatermarkPosition = C.pointer(pos)
        c.MaxTargetDimensions = C.pointer(dims)
        c.MaxFiltersCount = cfg.max_filters
        c.AllowExperiments = 1 if cfg.allow_experiments else 0
        if cfg.watermark is not None:
            wm = np.ascontiguousarray(cfg.watermark)
            h, w, ch = wm.shape
            step = (w * ch + 3) & ~3                       # cvCreateImage row alignment, as PrepareWatermark records it
            padded = np.zeros((h, step), np.uint8)
            padded[:, :w * ch] = wm.reshape(h, w * ch)
            ri = _RecoverInfo(_CvSize(w, h), 8, ch, step, step * h, padded.ctypes.data)
            keep += [padded, ri]
            c.WatermarkInfo = C.pointer(ri)
        keep.append(c)
        return c, keep

    # -- operators (bridge.h:4-7, filters.h:1) ------------------------------------------------------
    @classmethod
    def filter(cls, img: np.ndarray, request: str, allow_experiments: bool = True):
        L = cls.lib()
        p = cls.new_image(img)
        pp = C.POINTER(IplImage)(p.contents)
        code = L.Filter(C.byref(pp), C.create_string_buffer(request.encode()), 1 if allow_experiments else 0)
        out = cls.to_numpy(pp)
        L.cvReleaseImage(C.byref(pp))
        return code, out

    @classmethod
    def crop(cls, img, args: str, gravity: Optional[str] = None):
        L = cls.lib()
        p = cls.new_image(img)
        pp = C.POINTER(IplImage)(p.contents)
        g = C.create_string_buffer(gravity.encode()) if gravity is not None else None
        code = L.Crop(C.byref(pp), C.create_string_buffer(args.encode()), g)
        out = cls.to_numpy(pp)
        L.cvReleaseImage(C.byref(pp))
        return code, out

    @classmethod
    def resize(cls, img, args: str, cfg: Optional[OracleConfig] = None, simple: bool = False):
        L = cls.lib()
        c, keep = cls.make_config(cfg or OracleConfig())
        p = cls.new_image(img)
        pp = C.POINTER(IplImage)(p.contents)
        code = L.Resize(C.byref(pp), C.create_string_buffer(args.encode()), C.byref(c), 1 if simple else 0)
        out = cls.to_numpy(pp)
        L.cvReleaseImage(C.byref(pp))
        return code, out

    @classmethod
    def watermark(cls, img, cfg: OracleConfig):
        L = cls.lib()
        c, keep = cls.make_config(cfg)
        p = cls.new_image(img)
        code = L.Watermark(p, C.byref(c))
        out = cls.to_numpy(p)
        cls.release(p)
        return code, out

    @classmethod
    def call_inplace(cls, fn: str, img, *args):
        """Call a void kernel of filters.h:22-32 / helpers.h:16-17 on a copy of img."""
        L = cls.lib()
        p = cls.new_image(img)
        getattr(L, fn)(p, *args)
        out = cls.to_numpy(p)
        cls.release(p)
        return out

    @classmethod
    def alpha_over(cls, dst, src, opacity: float, x0: int = 0, y0: int = 0):
        L = cls.lib()
        d, s = cls.new_image(dst), cls.new_image(src)
        if x0 or y0:
            L.cvSetImageROI.argtypes = [C.c_void_p, C.c_int * 4]
            L.cvSetImageROI(d, (C.c_int * 4)(x0, y0, src.shape[1], src.shape[0]))
        L.AlphaBlendOver(d, s, C.c_float(opacity))
        out = cls.to_numpy(d)
        cls.release(d); cls.release(s)
        return out

    @classmethod
    def ascii(cls, img, args: str = "") -> bytes:
        """The reference's ASCII (filters.c:486-522); it converts its copy of the frame to HSV in place."""
        class _Memory(C.Structure):
            _fields_ = [("Buffer", C.c_void_p), ("Length", C.c_long), ("Error", C.c_int)]
        L = cls.lib()
        L.ASCII.restype = _Memory
        L.ASCII.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p]
        p = cls.new_image(img)
        m = L.ASCII(p, args.encode(), None)
        out = C.string_at(m.Buffer, m.Length)
        cls.release(p)
        return out

    @classmethod
    def perceived_brightness(cls, img) -> float:
        L = cls.lib()
        p = cls.new_image(img)
        v = float(L.CalcPerceivedBrightness(p))
        cls.release(p)
        return v

    @classmethod
    def run_job(cls, query: str, img: np.ndarray, cfg: Optional[OracleConfig] = None, exten: str = "png"):
        """RunJob (bridge.c:302-724) on a RAW-coded blob. Returns (code, step, image or None)."""
        L = cls.lib()
        cfg = cfg or OracleConfig()
        c, keep = cls.make_config(cfg)
        img = np.ascontiguousarray(_as3(img))
        h, w, ch = img.shape
        cap = max(w * h * 4, cfg.max_w * cfg.max_h * 4, 1 << 20) * 2
        out = np.empty(cap, np.uint8)
        ow, oh, oc, step, mime = (C.c_int(0) for _ in range(5))
        uri = ("/img." + exten + "?" + query).encode()
        code = L.ref_run_job(uri, exten.encode(), C.c_void_p(img.ctypes.data), w, h, ch, C.byref(c),
                             C.c_void_p(out.ctypes.data), C.c_long(cap), C.byref(ow), C.byref(oh), C.byref(oc),
                             C.byref(step), C.byref(mime))
        res = None
        if code == 0 and ow.value:
            res = out[:ow.value * oh.value * oc.value].reshape(oh.value, ow.value, oc.value).copy()
        return code, step.value, res

    # -- advancedio.c (compiled unmodified over oracle/fake_freeimage.c) ------------------------------------
    FIF_BMP, FIF_JPEG, FIF_TARGA, FIF_GIF = 0, 2, 17, 25

    @staticmethod
    def gif_container(frames) -> bytes:
        """The fake multi-page container fake_freeimage.c decodes. frames: dicts with `indices` (h x w uint8, TOP-DOWN),
        `palette` (256x4 B,G,R,x), left, top, dispose, key (-1 = none), time."""
        import struct
        out = [b"IMPGIF1\0", struct.pack("<i", len(frames))]
        for f in frames:
            idx = np.ascontiguousarray(f["indices"], np.uint8)
            h, w = idx.shape
            out.append(struct.pack("<7i", w, h, f.get("left", 0), f.get("top", 0), f.get("dispose", 0), f.get("key", -1), f.get("time", 0)))
            out.append(np.ascontiguousarray(f["palette"], np.uint8).tobytes())
            out.append(idx.tobytes())
        return b"".join(out)

    @staticmethod
    def fi_page_bits(indices_top_down: np.ndarray) -> np.ndarray:
        """The page's pixel block as FreeImage holds it (and as LoadGIF reads it): bottom-up scanlines, rows padded to
        4 bytes with zeros. Returns an (h, pitch) array; row 0 = bottom scanline."""
        idx = np.ascontiguousarray(indices_top_down, np.uint8)
        h, w = idx.shape
        bits = np.zeros((h, (w + 3) & ~3), np.uint8)
        bits[:, :w] = idx[::-1]
        return bits

    @classmethod
    def fi_load(cls, blob: bytes, fmt: int, destructive: bool = False, page: int = -1):
        """FiLoadFrames (advancedio.c:311-339). Returns (error, [dict(image, time, dispose, key)])."""
        L = cls.lib()
        L.ref_fi_load.restype = C.c_void_p
        L.ref_fi_load.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.ref_album_frame.argtypes = [C.c_void_p, C.c_int] + [C.POINTER(C.c_int)] * 6 + [C.c_void_p]
        L.ref_album_free.argtypes = [C.c_void_p]
        count, err = C.c_int(0), C.c_int(0)
        album = L.ref_fi_load(blob, len(blob), fmt, 1 if destructive else 0, page, C.byref(count), C.byref(err))
        frames = []
        if not err.value:
            for i in range(count.value):
                w, h, c, t, d, k = (C.c_int(0) for _ in range(6))
                if L.ref_album_frame(album, i, C.byref(w), C.byref(h), C.byref(c), C.byref(t), C.byref(d), C.byref(k), None):
                    break
                img = np.empty((h.value, w.value, c.value), np.uint8)
                L.ref_album_frame(album, i, C.byref(w), C.byref(h), C.byref(c), C.byref(t), C.byref(d), C.byref(k), C.c_void_p(img.ctypes.data))
                frames.append(dict(image=img, time=t.value, dispose=d.value, key=k.value))
        L.ref_album_free(album)
        return err.value, frames

    @classmethod
    def fi_save(cls, img: np.ndarray, fmt: int):
        """FiSaveFrames -> SaveSingle -> IplToFI32 / IplToFI24 (advancedio.c:65-101, 421-446) through the fake encoder.
        Returns (error, bpp, bits) with bits = the FIBITMAP's rows as they lie in memory (row 0 = bottom), pad removed."""
        import struct
        L = cls.lib()
        L.ref_fi_save.restype = C.c_long
        L.ref_fi_save.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_long, C.POINTER(C.c_int)]
        a = np.ascontiguousarray(img)
        h, w, c = a.shape
        cap = 64 + ((w * 4 + 3) & ~3) * h
        out = np.empty(cap, np.uint8)
        err = C.c_int(0)
        n = L.ref_fi_save(C.c_void_p(a.ctypes.data), w, h, c, a.strides[0], fmt, C.c_void_p(out.ctypes.data), cap, C.byref(err))
        if err.value or n < 24:
            return err.value, 0, None
        assert out[:8].tobytes() == b"IMPFI01\0"
        fw, fh, bpp, pitch = struct.unpack("<4i", out[8:24].tobytes())
        bits = out[24:24 + pitch * fh].reshape(fh, pitch)[:, :fw * bpp // 8].reshape(fh, fw, bpp // 8).copy()
        return 0, bpp, bits

    @classmethod
    def run_job_blob(cls, query: str, blob: bytes, cfg: Optional[OracleConfig] = None, exten: str = "gif"):
        """RunJob (bridge.c:302-724) on an arbitrary blob — the fake GIF container goes through the reference's own
        FiLoadFrames. Returns (code, step, image or None): the image decoded from cvEncodeImage's RAW container
        (format=png/jpg) or from SaveSingle's FIBITMAP dump (format=bmp...: rows bottom-up, as IplToFI32/24 wrote them)."""
        import struct
        L = cls.lib()
        cfg = cfg or OracleConfig()
        c, keep = cls.make_config(cfg)
        cap = max(cfg.max_w * cfg.max_h * 4, len(blob) * 8, 1 << 22)
        out = np.empty(cap, np.uint8)
        n, step, mime = C.c_long(0), C.c_int(0), C.c_int(0)
        uri = ("/img." + exten + "?" + query).encode()
        L.ref_run_job_blob.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.c_long, C.c_void_p, C.c_void_p, C.c_long,
                                       C.POINTER(C.c_long), C.POINTER(C.c_int), C.POINTER(C.c_int)]
        code = L.ref_run_job_blob(uri, exten.encode(), blob, len(blob), C.byref(c), C.c_void_p(out.ctypes.data), cap,
                                  C.byref(n), C.byref(step), C.byref(mime))
        img = None
        raw = out[:n.value].tobytes()
        cls.last_raw = raw                      # the encoded bytes as RunJob returned them (e.g. the multi-page container)
        if code == 0 and raw[8:12] == b"IMPR":
            w, h, ch = struct.unpack("<3i", raw[12:24])
            img = np.frombuffer(raw, np.uint8, w * h * ch, 24).reshape(h, w, ch).copy()
        elif code == 0 and raw[:8] == b"IMPFI01\0":
            w, h, bpp, pitch = struct.unpack("<4i", raw[8:24])
            img = np.frombuffer(raw, np.uint8, pitch * h, 24).reshape(h, pitch)[:, :w * bpp // 8].reshape(h, w, bpp // 8).copy()
        return code, step.value, img


class RefGpu(Ref):
    """The reference with INTEGRATION.md's edits applied (oracle/make_gpu_bridge.py): its own RunJob, FiLoadFrames and
    encoders, but steps 3-7 call imp_Crop / imp_Resize / imp_Filter / imp_Watermark / imp_BlendWithPaper + imp_FlushAll of
    libimp_gpu.so. Needs a GPU at run time; `available()` only says the prebuilt library travels with the repo."""
    _lib = None
    _cbs = None
    _started = False

    @classmethod
    def path(cls):
        return os.path.join(HERE, "_ref", "libimp_ref_gpu.so")

    @classmethod
    def available(cls) -> bool:
        return os.path.exists(cls.path())

    @classmethod
    def lib(cls):
        L = super().lib()
        if not cls._started:
            L.OnEnvStart()                # bridge.c:10 with the edit: imp_gpu_init(0) + the frame allocator
            cls._started = True
        return L
