"""CPU tests of the launch choice the planner stores with every pass (ImpHostPass::tiled / ::fallback, imp_pass_launches in
imp_planner.cpp): which kernel a job of the pass runs, its parameter, the op-interpreter flavour, the CTAs per job, the
dynamic shared memory and the occupancy class. A job whose source rows are 16-byte addressable takes `tiled`, any other
job `fallback`; the runtime only makes that one decision per job."""
import ctypes as C

import numpy as np
import pytest

from ngx_http_imgproc_b200 import api
from test_planner_host import REQS

# ImpKernel (imp_internal.h)
BLUR_GENERIC, DIRECT, STRIP, BLUR_TILE, CUBIC_RUN, CUBIC_TILE, GATHER_TILE = -1, 0, 1, 2, 3, 4, 5
SMEM_OPTIN = 200 * 1024
G_COPY, G_NN, G_AREA_INT, G_AREA_FRAC, G_CUBIC, G_LINEAR, G_BLUR = range(7)


@pytest.fixture(scope="module")
def launches(hostsim):
    """launches(w, h, c, cfgkw, **req) -> [(kind, tiled, fallback)] per pass; tiled / fallback =
    (kernel, param, flavour, ctas_per_job, smem_bytes, ctas_per_sm)."""
    lib = hostsim.lib
    lib.hostsim_plan_launch.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int)]
    lib.hostsim_plan_launch.restype = None

    def run(w, h, c, cfgkw, **req):
        ccfg, keep1 = api.Config(**cfgkw).to_c()
        creq, keep2 = api.make_request(**req)
        plan, step = C.c_void_p(), C.c_int(-1)
        rc = lib.hostsim_plan_create(C.byref(creq), C.byref(ccfg), w, h, c, C.byref(plan), C.byref(step))
        if rc:
            return None
        try:
            out = []
            for k in range(lib.hostsim_plan_passes(plan)):
                t, f = (C.c_int * 6)(), (C.c_int * 6)()
                lib.hostsim_plan_launch(plan, k, 1, t)
                lib.hostsim_plan_launch(plan, k, 0, f)
                out.append((lib.hostsim_plan_pass_kind(plan, k), tuple(t), tuple(f)))
            return out
        finally:
            lib.hostsim_plan_destroy(plan)
    return run


def _wm(w, h):
    return np.zeros((h, w, 4), np.uint8)


BASE = dict(max_w=0, max_h=0, max_filters=8, allow_experiments=True)
SEPIA = ["modulate=0,0,100", "colorize=704214,0.6"]
WM2 = dict(BASE, watermark=_wm(256, 64), wm_gravity_x="r", wm_gravity_y="b", wm_offset_x=10, wm_offset_y=10, wm_opacity=60)
WM5 = dict(BASE, watermark=_wm(64, 64), wm_gravity_x="r", wm_gravity_y="b", wm_offset_x=8, wm_offset_y=8, wm_opacity=100)

# (source w, h, c), config, request, tiled, fallback: the benchmark's shapes, one pass each
BENCH = {
    "cfg1": ((1920, 1080, 3), BASE, dict(resize="640,360"), (STRIP, 7, 1, 20, 53952, 4), (DIRECT, 0, 0, 240, 16, 0)),
    "cfg1l": ((1920, 1080, 3), BASE, dict(resize="640,360", interp=1), (STRIP, 7, 1, 20, 49472, 4), (DIRECT, 0, 0, 240, 16, 0)),
    "cfg2": ((3840, 2160, 4), WM2, dict(crop="3600px,2025px,c,c", resize="800,450"), (STRIP, 3, 2, 25, 67520, 3), (DIRECT, 0, 0, 375, 64, 0)),
    "cfg3": ((480, 270, 4), BASE, dict(resize="960,540,up", filters=SEPIA), (CUBIC_TILE, 64, 1, 135, 50944, 0), (CUBIC_RUN, 0, 0, 270, 832, 0)),
    "cfg3nn": ((480, 270, 4), BASE, dict(resize="960,540,up", filters=SEPIA, simple=True), (GATHER_TILE, 64, 1, 34, 13376, 0), (DIRECT, 0, 0, 510, 832, 0)),
    "cfg4": ((4000, 3000, 3), BASE, dict(filters=["blur=2.3", "vignette=0.8", "rotate=90"]), (BLUR_TILE, 6, 1, 5875, 39488, 0), (BLUR_GENERIC, 0, 0, 0, 64, 0)),
    "cfg5": ((1111, 777, 3), WM5, dict(resize="256,256"), (STRIP, 6, 2, 8, 73280, 3), (DIRECT, 0, 0, 64, 64, 0)),
    "blur6": ((800, 600, 3), BASE, dict(filters=["blur=6"]), (BLUR_GENERIC, 0, 0, 0, 16, 0), (BLUR_GENERIC, 0, 0, 0, 16, 0)),
    "rotate90": ((800, 600, 3), BASE, dict(filters=["rotate=90"]), (GATHER_TILE, 64, 1, 33, 40640, 0), (DIRECT, 0, 0, 475, 16, 0)),
}


@pytest.mark.parametrize("name", list(BENCH))
def test_bench_shapes(launches, name):
    (w, h, c), cfgkw, req, tiled, fallback = BENCH[name]
    passes = launches(w, h, c, cfgkw, **req)
    assert passes is not None and len(passes) == 1, passes
    _, t, f = passes[0]
    assert t == tiled, (name, t)
    assert f == fallback, (name, f)


def test_every_pass_has_a_launch_of_its_kind(launches):
    """Over the planner's request matrix: the fallback is the kind's general kernel, the tiled choice a kernel that serves
    the kind and fits the shared memory the tile kernels are configured for."""
    fallback_of = {G_CUBIC: CUBIC_RUN, G_BLUR: BLUR_GENERIC}
    tiles_of = {G_COPY: {GATHER_TILE}, G_NN: {GATHER_TILE}, G_AREA_INT: {STRIP}, G_AREA_FRAC: {STRIP},
                G_CUBIC: {CUBIC_TILE}, G_LINEAR: {STRIP, GATHER_TILE}, G_BLUR: {BLUR_TILE}}
    seen = set()
    for (h, w, c) in [(60, 80, 3), (45, 64, 4), (33, 47, 1), (480, 640, 3)]:
        for rq in REQS + [dict(filters=["blur=6"])]:
            for kind, t, f in launches(w, h, c, dict(BASE, max_filters=5), **rq) or []:
                assert f[0] == fallback_of.get(kind, DIRECT), (rq, kind, f)
                assert t == f or t[0] in tiles_of[kind], (rq, kind, t)
                assert t[4] <= SMEM_OPTIN and t[3] >= 0, (rq, t)
                seen.add(t[0])
    assert {STRIP, BLUR_TILE, CUBIC_TILE, GATHER_TILE, BLUR_GENERIC} <= seen, seen
