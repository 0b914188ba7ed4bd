"""Fractional INTER_AREA with exact integer taps (imp_planner.cpp area_exact, the strip kernel's MODE 2 in imp_tiles.cuh).

With the scale p/q per axis in lowest terms every weight is k/p, so an output pixel is N/D with N = sum k_y k_x S and
D = p_x p_y. The planner admits a pass only when D is odd, D <= 257 and its error bound shows that cvRound of the float sum
is round(N/D) = (N + (D-1)/2) / D, and the kernel then sums integers.

CPU: which scales qualify; the integer formula over the planner's tables equals imp_gather_area_frac (the float path the
other tests pin to OpenCV) on random, constant and near-tie frames, where N mod D is (D-1)/2 or (D+1)/2; the division by
the header's magic. GPU: the new mode bit-exact against the oracle over channels, op flavours, orientations, every tap
count the rule admits, cfg2 at full size and the near-tie frames; the same cases over the debug build."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import kernel_cases as K
from ngx_http_imgproc_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G_AREA_FRAC = 3


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("areashim") / "libarea_shim.so")
    cuda_inc = os.environ.get("CUDA_HOME", "/usr/local/cuda") + "/include"
    d = os.path.join(ROOT, "tests", "hostsim")
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-w", "-I" + cuda_inc, "-o", so,
                    os.path.join(d, "area_exact_shim.cpp"), os.path.join(d, "hostsim.cpp"),
                    os.path.join(ROOT, "ngx_http_imgproc_b200", "csrc", "imp_planner.cpp"), "-lm"], check=True)
    lib = C.CDLL(so)
    lib.hostsim_plan_create.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_int)]
    lib.hostsim_plan_destroy.argtypes = [C.c_void_p]
    lib.shim_area_info.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    lib.shim_area_info.restype = None
    lib.shim_area_tables.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 4 + [C.c_int, C.c_int]
    lib.shim_area_float.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
    return lib


class Pass:
    """Pass 0 of the plan of `req` on an h x w x c frame: header fields and, when exact, the integer tables."""

    def __init__(self, shim, shape, req, cfgkw=None):
        h, w, c = shape
        self.shim, self.shape = shim, shape
        ccfg, self._k1 = api.Config(**(cfgkw or K.BASE_KW)).to_c()
        creq, self._k2 = api.make_request(**req)
        plan, step = C.c_void_p(), C.c_int(-1)
        assert shim.hostsim_plan_create(C.byref(creq), C.byref(ccfg), w, h, c, C.byref(plan), C.byref(step)) == 0, req
        self.plan = plan
        v = (C.c_longlong * 13)()
        shim.shim_area_info(plan, 0, v)
        (self.kind, self.sc, self.sw, self.sh, self.bw, self.bh, self.max_xtaps, self.max_ytaps,
         self.D, self.bias, self.magic, self.nxt, self.nyt) = list(v)

    def close(self):
        self.shim.hostsim_plan_destroy(self.plan)

    def weights(self):
        """Dense integer weight matrices Wy (bh x sh) and Wx (bw x sw): N = Wy @ S @ Wx.T per channel."""
        xr = np.zeros((self.bw, 2), np.int32); yr = np.zeros((self.bh, 2), np.int32)
        xk = np.zeros((self.nxt, 2), np.int32); yk = np.zeros((self.nyt, 2), np.int32)
        assert self.shim.shim_area_tables(self.plan, 0, xr.ctypes.data, yr.ctypes.data, xk.ctypes.data, yk.ctypes.data, self.nxt, self.nyt) == 0
        Wx = np.zeros((self.bw, self.sw), np.int64); Wy = np.zeros((self.bh, self.sh), np.int64)
        for W, r, k in ((Wx, xr, xk), (Wy, yr, yk)):
            for d, (first, n) in enumerate(r):
                for si, kk in k[first:first + n]:
                    W[d, si] += kk
        return Wy, Wx

    def float_out(self, img):
        img = np.ascontiguousarray(img)
        out = np.zeros((self.bh, self.bw, self.sc), np.uint8)
        assert self.shim.shim_area_float(self.plan, 0, img.ctypes.data, img.strides[0], out.ctypes.data) == 0
        return out


def exact_out(Wy, Wx, D, win):
    """(N + (D-1)/2) // D over the window's pixels, per channel."""
    out = np.stack([Wy @ win[:, :, c].astype(np.int64) @ Wx.T for c in range(win.shape[2])], axis=2)
    return (out + (D - 1) // 2) // D, out


def near_tie(Wy, Wx, D, win, seed):
    """The window with one owned source pixel per output pixel (one that no other output reads) set so that N mod D is
    (D-1)/2 or (D+1)/2, where such a value exists. Returns the frame and the fraction of outputs that hit a tie residue."""
    win = win.copy()
    rng = np.random.default_rng(seed)

    def owned(W):
        used = (W > 0).sum(0)
        return np.array([max(np.nonzero((W[d] > 0) & (used == 1))[0], key=lambda s: W[d, s]) for d in range(W.shape[0])])
    oy, ox = owned(Wy), owned(Wx)
    wgt = Wy[np.arange(len(oy)), oy][:, None] * Wx[np.arange(len(ox)), ox][None, :]
    s = np.arange(256)
    for c in range(win.shape[2]):
        cur = win[np.ix_(oy, ox, [c])][:, :, 0].astype(np.int64)
        N = Wy @ win[:, :, c].astype(np.int64) @ Wx.T
        rest = N - wgt * cur
        r = (rest[:, :, None] + wgt[:, :, None] * s[None, None, :]) % D
        ok = (r == (D - 1) // 2) | (r == (D + 1) // 2)
        # among the tie values pick one at random, so that both residues and many pixel values occur
        score = np.where(ok, rng.random(ok.shape), -1.0)
        best = score.argmax(2)
        new = np.where(ok.any(2), best, cur)
        win[np.ix_(oy, ox, [c])] = new[:, :, None].astype(np.uint8)
    _, N = exact_out(Wy, Wx, D, win)
    hit = np.isin(N % D, [(D - 1) // 2, (D + 1) // 2]).mean()
    return win, hit


# ---- qualification ---------------------------------------------------------------------------------------------
QUALIFY = [
    ("cfg2", (2160, 3840, 4), dict(crop="3600px,2025px,c,c", resize="800,450"), 81),
    ("2.5x", (50, 100, 3), dict(resize="40,20"), 25),
    ("4.5x_by_1.5x", (27, 144, 4), dict(resize="32,18"), 27),
    ("1.5x_by_4.5x", (81, 48, 1), dict(resize="32,18"), 27),
    ("1x_by_2.5x", (100, 64, 4), dict(resize="64,40"), 5),
    ("11.5x_by_1.5x", (60, 920, 3), dict(resize="80,40"), 69),
    ("5/3", (50, 100, 4), dict(resize="60,30"), 25),
]
REFUSE = [
    ("1.6x", (80, 80, 4), dict(resize="50,50")),               # p = 8: D even
    ("8.5x_both", (170, 170, 4), dict(resize="20,20")),         # D = 17 * 17 = 289 > 257
    ("4.5x_by_1.6x", (80, 144, 4), dict(resize="32,50")),       # x qualifies, y (p = 8) does not
    ("1.5x_by_2x", (40, 48, 4), dict(resize="32,20")),          # an integer y scale of 2: p_y = 2
]


@pytest.mark.parametrize("name,shape,req,D", QUALIFY, ids=[q[0] for q in QUALIFY])
def test_qualifying_scales(shim, name, shape, req, D):
    p = Pass(shim, shape, req)
    try:
        assert p.kind == G_AREA_FRAC and p.D == D and p.bias == (D - 1) // 2 and p.magic == -(-(1 << 32) // D), (name, p.D)
    finally:
        p.close()


@pytest.mark.parametrize("name,shape,req", REFUSE, ids=[q[0] for q in REFUSE])
def test_refused_scales(shim, name, shape, req):
    p = Pass(shim, shape, req)
    try:
        assert p.kind == G_AREA_FRAC and p.D == 0, (name, p.D)
    finally:
        p.close()


def test_cfg5_shapes_stay_float(shim):
    """bench.py's cfg5 pool (512 sources to 256x256) keeps the float taps but for one source, 768x504 (3 x 63/32: D = 189,
    whose bound holds)."""
    rng = np.random.default_rng(6)
    shapes = [(int(rng.integers(240, 1537)), int(rng.integers(320, 2049)), 3 if rng.random() < 0.75 else 4) for _ in range(512)]
    exact = []
    for shape in shapes:
        p = Pass(shim, shape, dict(resize="256,256"), dict(K.BASE_KW))
        try:
            if p.kind == G_AREA_FRAC and p.D:
                exact.append((shape, p.D))
        finally:
            p.close()
    assert exact == [((504, 768, 4), 189)], exact


def test_magic_division():
    for D in range(3, 258, 2):
        magic = -(-(1 << 32) // D)
        n = np.arange(255 * D + (D - 1) // 2 + 1, dtype=np.uint64)
        assert np.array_equal((n * np.uint64(magic)) >> np.uint64(32), n // np.uint64(D)), D


# ---- the integer formula against the float path ----------------------------------------------------------------------
FORMULA = [(name, shape, req) for name, shape, req, _ in QUALIFY if name != "cfg2"] + [("cfg2_small", (81, 144, 4), dict(resize="32,18"))]


@pytest.mark.parametrize("sc", [1, 3, 4])
@pytest.mark.parametrize("name,shape,req", FORMULA, ids=[f[0] for f in FORMULA])
def test_integer_formula_equals_float_path(shim, name, shape, req, sc):
    h, w, _ = shape
    p = Pass(shim, (h, w, sc), req)
    try:
        assert p.D > 0, name
        Wy, Wx = p.weights()
        assert (Wx.sum(1) == Wx.sum(1)[0]).all() and (Wy.sum(1) == Wy.sum(1)[0]).all()
        assert Wx.sum(1)[0] * Wy.sum(1)[0] == p.D
        rng = np.random.default_rng(sum(map(ord, name)) + sc)
        frames = [rng.integers(0, 256, (h, w, sc), dtype=np.uint8), np.zeros((h, w, sc), np.uint8), np.full((h, w, sc), 255, np.uint8)]
        for seed in range(4):
            img = rng.integers(0, 256, (h, w, sc), dtype=np.uint8)
            tie, hit = near_tie(Wy, Wx, p.D, img, seed)
            assert hit > 0.5, (name, sc, hit)
            frames.append(tie)
        for i, img in enumerate(frames):
            want, _ = exact_out(Wy, Wx, p.D, img)
            got = p.float_out(img)
            assert want.max() <= 255
            assert np.array_equal(got, want.astype(np.uint8)), (name, sc, i, int((got != want).sum()))
    finally:
        p.close()


# ---- GPU ---------------------------------------------------------------------------------------------------------
def gpu_cases():
    """Every tap count 1..12 the rule admits (x scale (2n-1)/2, or 1 for n = 1; y scale (2m-1)/2), per source channels and
    op-interpreter flavour, the eight orientations in turn."""
    out = []
    i = 0
    bw, bh = 40, 70
    for sc in (1, 3, 4):
        for fl in (0, 1, 2):
            for n in range(1, 13):
                cfg, ops = K._flavour(fl, n)
                m = 2 + (n + sc + fl) % 5
                w = bw if n == 1 else bw * (2 * n - 1) // 2
                h = bh * (2 * m - 1) // 2
                out.append(K.Case(f"exact{n}_y{2 * m - 1}_c{sc}_fl{fl}", (h, w, sc), cfg, dict(resize=f"{bw},{bh}", filters=ops + K.ORIENT[i % 8]),
                                  ("strip", "area_frac", n, sc, fl)))
                i += 1
    return out


CFG2_KW = dict(K.BASE_KW, watermark=K.rnd_image(23, 64, 256, 4), wm_gravity_x="r", wm_gravity_y="b", wm_offset_x=10, wm_offset_y=10, wm_opacity=60)


def test_gpu_cases_take_the_exact_mode(shim, hostsim):
    for case in gpu_cases():
        p = Pass(shim, case.shape, case.req, case.cfgkw)
        try:
            assert p.D > 0 and p.max_xtaps == case.branch[2], (case.name, p.D, p.max_xtaps)
        finally:
            p.close()
        assert any(K.branch_key(b) == case.branch for b in K.plan_branches(hostsim, case)), case.name


def _check(gpu, orc, case, img):
    from test_kernel_branches import _assert_same, run_case_gpu
    from test_planner_host import _oracle
    code, _, ref = _oracle(orc, img, case.req, case.cfgkw)
    assert code == 0, case.name
    _assert_same(run_case_gpu(gpu, case, img), ref, case)


@pytest.mark.gpu
def test_exact_mode_matches_oracle(gpu, orc):
    for case in gpu_cases():
        _check(gpu, orc, case, case.image())


@pytest.mark.gpu
def test_cfg2_full_size_with_watermark(gpu, orc):
    case = K.Case("cfg2_full", (2160, 3840, 4), CFG2_KW, dict(crop="3600px,2025px,c,c", resize="800,450"), None)
    _check(gpu, orc, case, K.rnd_image(5, 2160, 3840, 4))


@pytest.mark.gpu
def test_near_tie_frames_on_the_gpu(gpu, orc, shim):
    for sc in (1, 3, 4):
        for name, shape, req in FORMULA:
            h, w, _ = shape
            p = Pass(shim, (h, w, sc), req)
            try:
                Wy, Wx = p.weights()
                img, _ = near_tie(Wy, Wx, p.D, np.random.default_rng(sc).integers(0, 256, (h, w, sc), dtype=np.uint8), sc)
            finally:
                p.close()
            _check(gpu, orc, K.Case(f"tie_{name}_c{sc}", (h, w, sc), K.WM_KW, dict(req, filters=["rotate=90"]), None), img)


@pytest.mark.gpu
def test_exact_mode_over_the_debug_build():
    """The GPU cases over libimp_gpu_dbg.so (-DIMP_DEBUG_BOUNDS: staged-tile offsets, tap-table indices, the accumulator
    bound) in a child process: no assertion fires and the outputs equal the oracle's."""
    dbg = os.path.join(ROOT, "ngx_http_imgproc_b200", "libimp_gpu_dbg.so")
    assert os.path.exists(dbg), "debug library not built (python -m ngx_http_imgproc_b200.build --debug)"
    code = r"""
import sys, ctypes as C
sys.path.insert(0, "."); sys.path.insert(0, "tests")
import ngx_http_imgproc_b200 as M
from oracle import oracle as O
import test_area_exact_int as T
L = M.library(); L.init(0)
L.lib.imp_gpu_debug_flags.restype = C.c_uint
n = 0
for case in T.gpu_cases():
    T._check(L, O, case, case.image())
    n += 1
flags = L.lib.imp_gpu_debug_flags()
print("BOUNDS", n, hex(flags))
assert flags == 0, hex(flags)
"""
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, IMP_GPU_LIB=dbg), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "BOUNDS" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]
    assert int(r.stdout.split("BOUNDS")[1].split()[0]) == len(gpu_cases())
