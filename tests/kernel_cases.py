"""The device code the planner can select, as a table of branches, and one small request per branch that lands on it.

A branch is what decides the instructions a job runs: the kernel (ImpKernel), its template arguments and the switch
inside it. The strip kernel (imp_tiles.cuh) picks its consumer per pass: fractional INTER_AREA switches on max_xtaps,
integer INTER_AREA on nx, each with cases 1..12; the blur tile kernel pads the effective tap radius to 3/6/9/12 with
zero taps, so every radius 1..12 is its own tap layout. Used by tests/test_kernel_branches.py (CPU: where each case
lands, through tests/hostsim; GPU: each case against the oracle)."""
import ctypes as C
from dataclasses import dataclass, field
from typing import Optional, Tuple

import numpy as np

from conftest import rnd_image, smooth_image
from ngx_http_imgproc_b200 import api

# ImpKernel (imp_internal.h), ImpGather (imp_plan.h)
BLUR_GENERIC, DIRECT, STRIP, BLUR_TILE, CUBIC_RUN, CUBIC_TILE, GATHER_TILE = -1, 0, 1, 2, 3, 4, 5
G_COPY, G_NN, G_AREA_INT, G_AREA_FRAC, G_CUBIC, G_LINEAR, G_BLUR = range(7)
KIND = {G_COPY: "copy", G_NN: "nn", G_AREA_INT: "area_int", G_AREA_FRAC: "area_frac", G_CUBIC: "cubic", G_LINEAR: "linear", G_BLUR: "blur"}
SMEM_OPTIN = 200 * 1024

# the eight output orientations (the dihedral group of the rectangle)
ORIENT = [[], ["flip=10"], ["flip=01"], ["rotate=180"], ["rotate=90"], ["rotate=270"], ["rotate=90", "flip=10"], ["rotate=90", "flip=01"]]

# op lists by op-interpreter flavour: 1 = no op or fused tables only, 2 = compositing + tables (a watermark), 0 = general
FL_OPS = {1: [[], ["gamma=1.3"]], 2: [[], ["gamma=0.8"]], 0: [["vignette=0.8"], ["modulate=60,70,80"]]}
WM = rnd_image(17, 9, 13, 4)
BASE_KW = dict(allow_experiments=True, max_filters=12, max_w=0, max_h=0)
WM_KW = dict(BASE_KW, watermark=WM, wm_gravity_x="r", wm_gravity_y="b", wm_offset_x=3, wm_offset_y=2, wm_opacity=70)


# ---- the branch table --------------------------------------------------------------------------------------------
def table():
    """Every branch the dispatch switches distinguish (keys as branch_key() returns them)."""
    t = set()
    for sc in (1, 3, 4):
        for fl in (0, 1, 2):
            for n in range(1, 13):
                t.add(("strip", "area_frac", n, sc, fl))
                t.add(("strip", "area_int", n, sc, fl))
            t.add(("strip", "linear", 0, sc, fl))
        for light in (0, 1):
            for kind in ("copy", "nn", "linear"):
                t.add(("gather", kind, sc, light))
            t.add(("cubic", sc, light))
        for kind in ("copy", "nn", "area_int", "area_frac", "cubic", "linear"):
            t.add(("direct", kind, sc))
        t.add(("cubic_run", sc))
    for sc in (3, 4):
        for r in range(1, 13):
            for nocomp in (0, 1):
                t.add(("blur", sc, r, nocomp))
        t.add(("blur_generic", sc))
    return t


# Branches no request reaches, each argued from the planner's code.
UNREACHABLE = {
    # imp_pass_launches: the fallback of an INTER_CUBIC pass is CubicRun, and its tile kernel is CubicTile; the direct
    # kernel's cubic instantiation only runs when IMP_GPU_FORCE_DIRECT=1 overrides the planner (test_gpu_parity covers it).
    ("direct", "cubic", 1): "cubic falls back to imp_cubic_run_kernel; imp_pass_kernel<CUBIC> only under IMP_GPU_FORCE_DIRECT",
    ("direct", "cubic", 3): "cubic falls back to imp_cubic_run_kernel; imp_pass_kernel<CUBIC> only under IMP_GPU_FORCE_DIRECT",
    ("direct", "cubic", 4): "cubic falls back to imp_cubic_run_kernel; imp_pass_kernel<CUBIC> only under IMP_GPU_FORCE_DIRECT",
}


def branch_key(b):
    """b: the dict plan_branches() gives for one pass."""
    k, kind, sc = b["kernel"], KIND[b["kind"]], b["sc"]
    if k == STRIP:
        n = b["max_xtaps"] if b["kind"] == G_AREA_FRAC else b["nx"] if b["kind"] == G_AREA_INT else 0
        return ("strip", kind, n, sc, b["flavour"])
    if k == GATHER_TILE:
        return ("gather", kind, sc, b["flavour"])
    if k == CUBIC_TILE:
        return ("cubic", sc, b["flavour"])
    if k == BLUR_TILE:
        return ("blur", sc, b["r_eff"], b["flavour"])
    if k == DIRECT:
        return ("direct", kind, sc)
    if k == CUBIC_RUN:
        return ("cubic_run", sc)
    return ("blur_generic", sc)


BRANCH_FIELDS = ["kind", "sc", "dc", "kernel", "flavour", "param", "max_xtaps", "nx", "ny", "gt", "blur_r", "r_eff",
                 "tile_rs", "tile_rows", "tile_smem", "smem_bytes"]


def plan_branches(hostsim, case, tiled=None):
    """Per pass of the case's plan, the fields of hostsim_plan_branch for the launch its jobs take: `tiled` when the
    source rows are 16-byte addressable (every pass but a first one read from a padded source), else `fallback`."""
    lib = hostsim.lib
    lib.hostsim_plan_branch.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int)]
    lib.hostsim_plan_branch.restype = None
    h, w, c = case.shape
    ccfg, keep1 = api.Config(**case.cfgkw).to_c()
    creq, keep2 = api.make_request(**case.req)
    plan, step = C.c_void_p(), C.c_int(-1)
    rc = lib.hostsim_plan_create(C.byref(creq), C.byref(ccfg), w, h, c, C.byref(plan), C.byref(step))
    assert rc == 0, (case.name, rc)
    try:
        out = []
        for k in range(lib.hostsim_plan_passes(plan)):
            v = (C.c_int * 16)()
            lib.hostsim_plan_branch(plan, k, int(tiled if tiled is not None else not (k == 0 and case.src_pad)), v)
            out.append(dict(zip(BRANCH_FIELDS, list(v))))
        return out
    finally:
        lib.hostsim_plan_destroy(plan)


# ---- cases -------------------------------------------------------------------------------------------------------
@dataclass
class Case:
    name: str
    shape: Tuple[int, int, int]          # source h, w, c
    cfgkw: dict
    req: dict
    branch: tuple                        # the branch the case is meant to land on (one of its passes)
    src_pad: int = 0                     # > 0: source rows src_pad bytes longer than w*c (pitch % 16 != 0: the fallback)
    expect: dict = field(default_factory=dict)   # other fields of that pass the case pins (ring stages, smem, ...)

    def image(self):
        h, w, c = self.shape
        seed = sum(map(ord, self.name)) % 1000
        return smooth_image(seed, h, w, c) if seed % 2 else rnd_image(seed, h, w, c)

    @property
    def vignette(self):
        return any("vignette" in f for f in self.req.get("filters", []))


def _flavour(fl, i):
    """(config, filters) of op-interpreter flavour fl; i picks between the two op lists of that flavour."""
    return (WM_KW if fl == 2 else BASE_KW), list(FL_OPS[fl][i % 2])


# Strip cases: 77 output columns (two full strips of 32 and a partial one), 139 output rows (17 tiles of 8 and a partial one:
# the ring of at most 8 stages wraps at least twice).
SW, SH = 77, 139
# fractional INTER_AREA with n x taps: source widths over 77 columns whose largest column has n taps; n = 1 is the
# unscaled axis, even n an integer x scale (every column n taps), odd n a fractional one (narrower columns: zero-weight
# padded taps). The y scale is fractional throughout.
FRAC_W = {n: 77 * n if n % 2 == 0 or n == 1 else round(77 * (n - 1.5)) for n in range(1, 13)}
FRAC_H = [209, 244, 181]


def strip_cases():
    out = []
    i = 0
    for sc in (1, 3, 4):
        for fl in (0, 1, 2):
            for n in range(1, 13):
                cfg, ops = _flavour(fl, n)
                h = FRAC_H[(n + sc) % 3]
                out.append(Case(f"frac{n}_c{sc}_fl{fl}", (h, FRAC_W[n], sc), cfg, dict(resize=f"{SW},{SH}", filters=ops + ORIENT[i % 8]),
                                ("strip", "area_frac", n, sc, fl)))
                i += 1
                ny = 2 if n == 1 else 1 + n % 3
                out.append(Case(f"int{n}x{ny}_c{sc}_fl{fl}", (SH * ny, SW * n, sc), cfg, dict(resize=f"{SW},{SH}", filters=ops + ORIENT[i % 8]),
                                ("strip", "area_int", n, sc, fl)))
                i += 1
            cfg, ops = _flavour(fl, sc)
            out.append(Case(f"linear_c{sc}_fl{fl}", (237, 131, sc), cfg, dict(resize=f"{SW},{SH}", interp=1, filters=ops + ORIENT[i % 8]),
                            ("strip", "linear", 0, sc, fl)))
            i += 1
    return out


# Blur: sigma whose Gaussian (SURVEY App. A.5) has effective tap radius r once zero outer taps are trimmed.
BLUR_SIGMA = {1: 0.45, 2: 0.75, 3: 1.1, 4: 1.45, 5: 1.8, 6: 2.15, 7: 2.55, 8: 2.9, 9: 3.25, 10: 3.6, 11: 3.9, 12: 4.3}


def tile_cases():
    out = []
    i = 0
    for sc in (1, 3, 4):
        for light in (0, 1):
            fl = 1 if light else 0
            cfg, ops = _flavour(fl, sc + i)
            if light == 0 and i % 2:
                cfg, ops = WM_KW, []                           # compositing alone clears LIGHT too
            out.append(Case(f"copy_c{sc}_l{light}", (101, 150, sc), cfg, dict(filters=ops + ORIENT[i % 8]), ("gather", "copy", sc, light)))
            i += 1
            out.append(Case(f"nn_c{sc}_l{light}", (67, 97, sc), cfg, dict(resize="150,101,up", simple=True, filters=ops + ORIENT[i % 8]),
                            ("gather", "nn", sc, light)))
            i += 1
            out.append(Case(f"linear_up_c{sc}_l{light}", (67, 97, sc), cfg, dict(resize="150,101,up", interp=1, filters=ops + ORIENT[i % 8]),
                            ("gather", "linear", sc, light)))
            i += 1
            out.append(Case(f"cubic_c{sc}_l{light}", (45, 67, sc), cfg, dict(resize="150,101,up", filters=ops + ORIENT[i % 8]),
                            ("cubic", sc, light)))
            i += 1
    for sc in (3, 4):
        for r in range(1, 13):
            for nocomp in (0, 1):
                cfg = BASE_KW if nocomp else WM_KW
                extra = ["gamma=1.2"] if (r + sc) % 3 == 0 else ["vignette=0.7"] if (r + sc) % 3 == 1 else []
                out.append(Case(f"blur_r{r}_c{sc}_nc{nocomp}", (97, 131, sc), cfg, dict(filters=[f"blur={BLUR_SIGMA[r]}"] + extra + ORIENT[i % 8]),
                                ("blur", sc, r, nocomp)))
                i += 1
    return out


def fallback_cases():
    """The kernels a pass falls back to: imp_pass_kernel per kind x source channels, imp_cubic_run_kernel, the two-launch
    Gaussian."""
    out = []
    for i, sc in enumerate((1, 3, 4)):
        o = ORIENT[(3 * i + 1) % 8]
        # a copy always fits the gather tile: only a source pitch that is not a multiple of 16 sends it to the direct kernel
        # (4-channel rows stay 4-byte addressable, as imp_gpu_run_device requires)
        out.append(Case(f"direct_copy_c{sc}", (61, 83, sc), BASE_KW, dict(filters=["gamma=1.1"] + o), ("direct", "copy", sc), src_pad=8 if sc == 4 else 5))
        out.append(Case(f"direct_nn_c{sc}", (150, 200, sc), BASE_KW, dict(resize="90,70", simple=True, filters=o), ("direct", "nn", sc)))
        out.append(Case(f"direct_int13_c{sc}", (30, 13 * 21, sc), BASE_KW, dict(resize="21,15", filters=o), ("direct", "area_int", sc)))
        out.append(Case(f"direct_frac13_c{sc}", (60, 13 * 21 - 7, sc), BASE_KW, dict(resize="21,37", filters=o), ("direct", "area_frac", sc)))
        out.append(Case(f"direct_linear_c{sc}", (1200, 1000, sc), BASE_KW, dict(resize="25,29", interp=1, filters=o), ("direct", "linear", sc)))
        out.append(Case(f"cubic_run_c{sc}", (900, 60, sc), BASE_KW, dict(resize="121,99,up", filters=o), ("cubic_run", sc)))
    for sc in (3, 4):
        out.append(Case(f"blur_generic_c{sc}", (97, 131, sc), BASE_KW, dict(filters=["blur=4.7", "rotate=90"]), ("blur_generic", sc)))
    return out


def cases():
    return strip_cases() + tile_cases() + fallback_cases()


# ---- footprint limits ----------------------------------------------------------------------------------------------
# Pairs that straddle each limit the planner keeps a tile kernel under (imp_planner.cpp): the first case takes the tile
# kernel at (or next to) the largest footprint it accepts, the second one just past it takes the smaller tile or the
# fallback. The largest footprint a kernel accepts is where its shared-memory indexing is most likely to break.
INT12 = dict(resize=f"{SW},{SH}")
GRADMAP = "gradmap=306090,eecc00"


def limit_pairs():
    """[(limit, inside case, outside case)]: the inside case lands on its branch (and the fields in `expect`), the outside
    case on the next smaller tile or the fallback."""
    P = [
        # strip, max_xtaps <= 12 (integer and fractional)
        ("strip_xtaps_int", ((SH * 2, SW * 12, 4), BASE_KW, dict(INT12, filters=["rotate=90"]), ("strip", "area_int", 12, 4, 1)),
                            ((SH * 2, SW * 13, 4), BASE_KW, dict(INT12, filters=["rotate=90"]), ("direct", "area_int", 4))),
        ("strip_xtaps_frac", ((181, FRAC_W[12], 4), BASE_KW, dict(INT12, filters=["flip=01"]), ("strip", "area_frac", 12, 4, 1)),
                             ((181, round(SW * 11.5), 4), BASE_KW, dict(INT12, filters=["flip=01"]), ("direct", "area_frac", 4))),
        # strip, 100 KB per stage (AREA): 12x8 on 4 channels is a 100 352-byte box, two ring stages, 200 896 bytes in all
        ("strip_100k", ((SH * 8, SW * 12, 4), BASE_KW, dict(INT12), ("strip", "area_int", 12, 4, 1), 0, dict(param=2, tile_smem=100352, smem_bytes=200896)),
                       ((SH * 9, SW * 12, 4), BASE_KW, dict(INT12), ("direct", "area_int", 4))),
        # strip, rows <= 256 (integer 1x32 against 1x33; fractional y scale near 32)
        ("strip_rows_int", ((SH * 32, SW, 1), BASE_KW, dict(INT12, filters=["rotate=270"]), ("strip", "area_int", 1, 1, 1), 0, dict(tile_rows=256)),
                           ((SH * 33, SW, 1), BASE_KW, dict(INT12, filters=["rotate=270"]), ("direct", "area_int", 1))),
        ("strip_rows_frac", ((4430, 116, 1), BASE_KW, dict(INT12, filters=["gamma=1.3"]), ("strip", "area_frac", 3, 1, 1), 0, dict(tile_rows=256)),
                            ((4435, 116, 1), BASE_KW, dict(INT12, filters=["gamma=1.3"]), ("direct", "area_frac", 1))),
        # integer strip, isx * isy <= 256
        ("strip_int_area", ((SH * 21, SW * 12, 1), WM_KW, dict(INT12), ("strip", "area_int", 12, 1, 2), 0, dict(param=2)),
                           ((SH * 22, SW * 12, 1), WM_KW, dict(INT12), ("direct", "area_int", 1))),
        # LINEAR strip: tile_rs <= 2048, 64 KB
        ("strip_linear_rs", ((209, 1246, 4), BASE_KW, dict(INT12, interp=1), ("strip", "linear", 0, 4, 1), 0, dict(tile_rs=2032)),
                            ((209, 1253, 4), BASE_KW, dict(INT12, interp=1), ("direct", "linear", 4))),
        ("strip_linear_64k", ((596, 1246, 4), BASE_KW, dict(INT12, interp=1, filters=["flip=10"]), ("strip", "linear", 0, 4, 1), 0, dict(tile_smem=65024)),
                             ((597, 1246, 4), BASE_KW, dict(INT12, interp=1, filters=["flip=10"]), ("direct", "linear", 4))),
        # LINEAR: scale 1.25 takes the gather tile kernel, beyond it the strip kernel
        ("linear_1.25", ((125, 125, 3), BASE_KW, dict(resize="100,100", interp=1, filters=["rotate=90"]), ("gather", "linear", 3, 1)),
                        ((126, 125, 3), BASE_KW, dict(resize="100,100", interp=1, filters=["rotate=90"]), ("strip", "linear", 0, 3, 1))),
        # gather tile: T = 64 up to 24 KB, then T = 32
        ("gather_24k", ((140, 151, 4), BASE_KW, dict(resize="150,101", simple=True, filters=["rotate=270"]), ("gather", "nn", 4, 1), 0, dict(gt=64, tile_smem=24208)),
                       ((140, 152, 4), BASE_KW, dict(resize="150,101", simple=True, filters=["rotate=270"]), ("gather", "nn", 4, 1), 0, dict(gt=32))),
        # NN staging: scale_y <= 1.5 and scale_x <= 2
        ("nn_scale_y", ((150, 100, 3), BASE_KW, dict(resize="100,100", simple=True, filters=["flip=11"]), ("gather", "nn", 3, 1)),
                       ((151, 100, 3), BASE_KW, dict(resize="100,100", simple=True, filters=["flip=11"]), ("direct", "nn", 3))),
        ("nn_scale_x", ((100, 200, 3), BASE_KW, dict(resize="100,100", simple=True), ("gather", "nn", 3, 1), 0, dict(gt=32)),
                       ((100, 201, 3), BASE_KW, dict(resize="100,100", simple=True), ("direct", "nn", 3))),
        # cubic: T = 64 / 32 / column runs at 52 KB (4 channels) and at 160 rows (1 channel)
        ("cubic_52k_64", ((57, 67, 4), BASE_KW, dict(resize="150,101,up"), ("cubic", 4, 1), 0, dict(gt=64)),
                         ((58, 67, 4), BASE_KW, dict(resize="150,101,up"), ("cubic", 4, 1), 0, dict(gt=32))),
        ("cubic_52k_32", ((215, 67, 4), BASE_KW, dict(resize="150,101,up", filters=["vignette=0.6"]), ("cubic", 4, 0), 0, dict(gt=32)),
                         ((216, 67, 4), BASE_KW, dict(resize="150,101,up", filters=["vignette=0.6"]), ("cubic_run", 4))),
        ("cubic_rows_64", ((250, 67, 1), BASE_KW, dict(resize="150,101,up"), ("cubic", 1, 1), 0, dict(gt=64, tile_rows=160)),
                          ((251, 67, 1), BASE_KW, dict(resize="150,101,up"), ("cubic", 1, 1), 0, dict(gt=32))),
        ("cubic_rows_32", ((508, 67, 1), BASE_KW, dict(resize="150,101,up", filters=["rotate=90"]), ("cubic", 1, 1), 0, dict(gt=32, tile_rows=160)),
                          ((509, 67, 1), BASE_KW, dict(resize="150,101,up", filters=["rotate=90"]), ("cubic_run", 1))),
        # blur: radius 12 is the largest tile (sigma ~4.3), radius 13 the two-launch Gaussian
        ("blur_radius", ((97, 131, 4), BASE_KW, dict(filters=["blur=4.3", "flip=10"]), ("blur", 4, 12, 1), 0, dict(blur_r=12)),
                        ((97, 131, 4), BASE_KW, dict(filters=["blur=4.6", "flip=10"]), ("blur_generic", 4))),
        # launch: the 200 KB opt-in; the 12x8 box with four gradmaps' tables still fits, five do not
        ("optin_200k", ((SH * 8, SW * 12, 4), BASE_KW, dict(INT12, filters=[GRADMAP] * 4), ("strip", "area_int", 12, 4, 0), 0, dict(smem_bytes=204224)),
                       ((SH * 8, SW * 12, 4), BASE_KW, dict(INT12, filters=[GRADMAP] * 5), ("direct", "area_int", 4))),
    ]
    return [(name, Case(f"{name}_in", *a), Case(f"{name}_out", *b)) for name, a, b in P]


def ring_cases():
    """The ring's two extremes: 8 stages (small boxes) and 2 (the largest)."""
    return [Case("ring8_int2x2_c1", (SH * 2, SW * 2, 1), BASE_KW, dict(INT12, filters=["flip=01"]), ("strip", "area_int", 2, 1, 1), 0, dict(param=8)),
            Case("ring8_frac1_c1", (209, SW, 1), BASE_KW, dict(INT12, filters=["rotate=90"]), ("strip", "area_frac", 1, 1, 1), 0, dict(param=8)),
            Case("ring2_int12x8_c4", (SH * 8, SW * 12, 4), WM_KW, dict(INT12, filters=["rotate=270"]), ("strip", "area_int", 12, 4, 2), 0, dict(param=2))]


def all_cases():
    """Every case once: one per branch, the limit pairs and the ring extremes."""
    out = cases() + ring_cases()
    for _, a, b in limit_pairs():
        out += [a, b]
    return out
