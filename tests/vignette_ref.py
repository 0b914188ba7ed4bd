"""High-precision reference of the vignette mask (filters.c:693-703 RadialGradient), CPU only.

For a vignette op whose frame is w x h with centre (cx, cy), the mask of a pixel depends only on (|dx|, |dy|) =
(|cx - x|, |cy - y|). The reference computes, per pixel,

    distance = (float) sqrt(dx*dx + dy*dy)                       exact squares, correctly rounded sqrt, narrowed
    raw      = (float)((float)(distance / maxr) * intensity)      IEEE float division and product
    mask     = (float) pow(cos((double) raw), 4)

The float steps are reproduced here in numpy with IEEE rounding. The double step is where implementations part: the
reference calls glibc's cos and pow, the device (imp_vignette_mask, imp_vignette_table_kernel) calls CUDA's double cos
and squares twice, the CPU build of the same code calls glibc's cos and squares twice. Each result is the true value
t = cos(raw)^4 times (1 + e) with a bounded e, and narrowing to float then gives the float nearest t unless a float
rounding boundary (the midpoint of two adjacent floats) lies within t * (1 +- e). Such an entry is "ambiguous": two
conforming implementations may disagree on it by one float ulp, which can move trunc(V * mask) by 1. Every other entry
is "exact": all of them must give round_to_float(t).

The bound e, from each function's documented maximum error (one double ulp is at most 2^-52 of the value):
  - glibc cos and pow: at most 1 ulp each (glibc manual, "Known Maximum Errors in Math Functions", x86_64).
    pow(C, 4) with C = cos(raw) (1 + a), |a| <= 2^-52, is C^4 (1 + b), |b| <= 2^-52:
        1 + e_ref <= (1 + 2^-52)^4 (1 + 2^-52)
  - CUDA double cos: at most 2 ulp (CUDA Math API, double precision functions). c2 = C*C and c2*c2 round to nearest,
    2^-53 each, and the second squaring doubles the first rounding:
        1 + e_dev <= (1 + 2^-51)^4 (1 + 2^-53)^2 (1 + 2^-53)
  - glibc cos with the two squarings (the CPU build of imp_vignette_mask):
        1 + e_host <= (1 + 2^-52)^4 (1 + 2^-53)^3
  The lower sides are the same products with minus signs and are smaller in magnitude. DELTA is the largest of the
  three, about 9.5 * 2^-52 = 2.1e-15; no slack is added to it.

The screen evaluates cos(raw)^4 in np.longdouble (64-bit significand, error far below 2^-56 of the value) and sends
every entry within DELTA + 2^-56 of a boundary to mpmath at 60 digits, which decides it.
"""
from dataclasses import dataclass

import mpmath
import numpy as np

MARGIN = 64                     # IMP_VIGNETTE_MARGIN (imp_plan.h): table entries beyond the frame in both directions
TABLE_LIMIT = 16 << 20          # the planner tabulates a frame's mask when (nx * ny) <= 16M entries, else per pixel

_DPS = 60
with mpmath.workdps(_DPS):
    _U = mpmath.mpf(2) ** -53                                   # unit roundoff of double: half an ulp, relative
    DELTA_REF = (1 + 2 * _U) ** 4 * (1 + 2 * _U) - 1
    DELTA_DEV = (1 + 4 * _U) ** 4 * (1 + _U) ** 3 - 1
    DELTA_HOST = (1 + 2 * _U) ** 4 * (1 + _U) ** 3 - 1
    DELTA = max(DELTA_REF, DELTA_DEV, DELTA_HOST)
_SCREEN = float(DELTA) + 2.0 ** -56


def table_dims(w, h, cx, cy):
    """(nx, ny): the |dx| and |dy| a frame's pixels and the margin reach (the planner's table size)."""
    return max(cx, w - 1 - cx) + MARGIN + 1, max(cy, h - 1 - cy) + MARGIN + 1


def raw_table(maxr, intensity, nx, ny):
    """float32 raw = (distance / maxr) * intensity for |dx| < nx, |dy| < ny, shape (ny, nx): the reference's float steps."""
    i = np.arange(nx, dtype=np.float64)
    j = np.arange(ny, dtype=np.float64)
    d2 = j[:, None] * j[:, None] + i[None, :] * i[None, :]          # exact: both < 2^26 squared stays below 2^53
    distance = np.sqrt(d2).astype(np.float32)
    return ((distance / np.float32(maxr)).astype(np.float32) * np.float32(intensity)).astype(np.float32)


def _bounds(f):
    """The rounding boundaries around float32 f: the midpoints with its two neighbours (float64, exact)."""
    f64 = f.astype(np.float64)
    lo = (f64 + np.nextafter(f, np.float32(-np.inf)).astype(np.float64)) / 2
    hi = (f64 + np.nextafter(f, np.float32(np.inf)).astype(np.float64)) / 2
    return lo, hi


@dataclass
class MaskClass:
    """mask: round_to_float(cos(raw)^4) per entry; ambiguous: entries a conforming implementation may round the other
    way; alt: the other candidate there (equal to mask elsewhere)."""
    mask: np.ndarray
    ambiguous: np.ndarray
    alt: np.ndarray

    @property
    def count(self):
        return int(self.ambiguous.sum())


def classify_raw(raw):
    """Classifies float32 arguments (any shape): returns MaskClass of the same shape."""
    assert np.finfo(np.longdouble).nmant >= 63, "the screen needs an extended long double"
    u, inv = np.unique(raw.ravel(), return_inverse=True)
    c = np.cos(u.astype(np.longdouble))
    c2 = c * c
    t = c2 * c2
    f = t.astype(np.float32)
    lo, hi = _bounds(f)
    tl = t.astype(np.longdouble)
    near = np.minimum(np.abs(tl - lo.astype(np.longdouble)), np.abs(hi.astype(np.longdouble) - tl)) <= _SCREEN * tl
    mask, amb, alt = f.copy(), np.zeros(u.shape, bool), f.copy()
    with mpmath.workdps(_DPS):
        for k in np.flatnonzero(near):
            mask[k], amb[k], alt[k] = decide(mpmath.cos(mpmath.mpf(float(u[k]))) ** 4)
    shape = raw.shape
    return MaskClass(mask[inv].reshape(shape), amb[inv].reshape(shape), alt[inv].reshape(shape))


def decide(t):
    """(float nearest t, ambiguous, the other candidate) for a value t given as an mpf of at least _DPS digits."""
    with mpmath.workdps(_DPS):
        f = np.float32(float(t))                    # t -> double -> float may round twice: settle it against t itself
        for g in (np.nextafter(f, np.float32(-np.inf)), np.nextafter(f, np.float32(np.inf))):
            if abs(mpmath.mpf(float(g)) - t) < abs(mpmath.mpf(float(f)) - t):
                f = g
        lo, hi = (float(b[0]) for b in _bounds(np.array([f], np.float32)))
        dlo, dhi = t - mpmath.mpf(lo), mpmath.mpf(hi) - t
        if min(dlo, dhi) <= DELTA * abs(t):
            return f, True, np.nextafter(f, np.float32(-np.inf) if dlo <= dhi else np.float32(np.inf))
        return f, False, f


_CACHE = {}


def classify(maxr, intensity, nx, ny):
    """MaskClass of the table mask[|dy|][|dx|], |dx| < nx, |dy| < ny, for one op (cached)."""
    key = (float(np.float32(maxr)), float(np.float32(intensity)), int(nx), int(ny))
    if key not in _CACHE:
        _CACHE[key] = classify_raw(raw_table(maxr, intensity, nx, ny))
    return _CACHE[key]


def frame_mask(op):
    """For a vignette op (a dict with cx, cy, maxr, intensity, w, h; see HostSim.vignette_ops): the float mask over the
    op's own w x h frame and the boolean image of its ambiguous pixels, both (h, w)."""
    w, h, cx, cy = op["w"], op["h"], op["cx"], op["cy"]
    nx, ny = table_dims(w, h, cx, cy)
    mc = classify(op["maxr"], op["intensity"], nx, ny)
    dy = np.abs(cy - np.arange(h))[:, None]
    dx = np.abs(cx - np.arange(w))[None, :]
    return mc.mask[dy, dx], mc.ambiguous[dy, dx]


def gray_expected(op, v):
    """The result of one vignette on a gray frame (b = g = r = v, so S = 0 and V = v): trunc(v * mask) per pixel, from the
    high-precision mask alone, plus the ambiguous pixels. v: (h, w) uint8 in the op's frame."""
    mask, amb = frame_mask(op)
    out = np.trunc(v.astype(np.float32) * mask).astype(np.int32) & 255    # NaN mask: low byte 0, as on x86
    return out.astype(np.uint8), amb
