"""Vignette against a high-precision mask (tests/vignette_ref.py). Every table entry whose float rounding no conforming
double implementation can change ("exact") must come out of the oracle, the CPU build of the kernels' code and the device
as round_to_float(cos(raw)^4); a result may differ from the reference by 1 only at pixels an ambiguous entry reaches.

CPU: the ambiguous entries of every vignette frame the suite uses and of a sweep of frame sizes, counted and printed; the
oracle's and hostsim's mask tables against the reference; the planner's table dimensions and the 16M-entry limit; gray
frames through hostsim against trunc(V * mask). GPU: gray frames against the reference mask alone, for every orientation
before and after the vignette, crops, 1 x N and N x 1 frames and every kernel family; the colour version against the
oracle; both sides of the table limit (the per-pixel device path); cfg4 at full size is in test_gpu_parity."""
import numpy as np
import pytest

import golden_util as G
import kernel_cases as K
import vignette_ref as VR
from conftest import rnd_image, smooth_image
from ngx_http_imgproc_b200 import api
from test_planner_host import REQS, _oracle

EXP = dict(allow_experiments=True, max_filters=12, max_w=0, max_h=0)
VIGS = ["vignette=0.8", "vignette=4,3", "vignette=0.5,0.7", "vignette=0.6", "vignette=0.7", "vignette=0.9,0.8", "vignette=,"]


def _vig_args(f):
    """(intensity, radius) of a vignette filter, by the oracle's grammar (oracle.apply_filter)."""
    from oracle import oracle as O
    t = O._tokens(f.split("=", 1)[1] if "=" in f else "")
    return (O.c_strtof(t[0]) if len(t) > 0 else 0.5), (O.c_strtof(t[1]) if len(t) > 1 else 1.0)


# ---- the requests of this module ---------------------------------------------------------------------------------------
# (source shape, request) pairs: odd and even frames, 1 x 1, 1 x N, N x 1, every orientation before the vignette (the op's
# frame differs from the base frame) and after it, crop windows, a resize of each family in front of it.
def matrix():
    out = []
    for k, (h, w) in enumerate([(1, 1), (1, 37), (41, 1), (2, 2), (48, 64), (49, 65), (77, 130), (131, 67), (240, 320)]):
        for oi, pre in enumerate(K.ORIENT):
            post = K.ORIENT[(oi + k) % 8] if oi % 2 else []
            out.append(((h, w, (3, 1, 4)[(oi + k) % 3]), dict(filters=pre + [VIGS[(oi + k) % 6]] + post)))
    for crop in ("61px,37px,5px,3px", "1px,90px,c,c", "90px,1px,r,b", "3,2", "77px,50px,c,c"):
        out.append(((97, 131, 3), dict(crop=crop, filters=["rotate=90", "vignette=0.8"])))
    for rq in (dict(resize="77,139"), dict(resize="150,101,up", simple=True), dict(resize="150,101,up", interp=1),
               dict(resize="150,101,up"), dict(resize="40,23", interp=1)):
        for oi in (0, 4, 7):
            out.append(((209, 231, 3), dict(rq, filters=K.ORIENT[oi] + ["vignette=0.6"] + K.ORIENT[(oi + 3) % 8])))
    out.append(((97, 131, 3), dict(filters=["blur=2.3", "vignette=0.8", "rotate=90"])))
    out.append(((97, 131, 3), dict(filters=["rotate=270", "blur=1.1", "vignette=4,3", "flip=01"])))
    return out


def kernel_family_cases():
    """The kernel_cases cases with a vignette and no compositing: one or more per kernel family (strip, gather, cubic, blur
    tile, the general kernels), partial tiles throughout."""
    return [c for c in K.all_cases() if c.vignette and "watermark" not in c.cfgkw and not c.req.get("pack") and not c.req.get("flatten")]


def suite_requests():
    """(source shape, config, request) of every vignette request the suite plans, as far as it is enumerable here."""
    rs = []
    for case in G.load():
        if "vignette" in case["query"] and case["code"] == 0:
            rs.append((case["img"].shape, case["cfgkw"], G.split_query(case["query"])))
    for case in K.all_cases():
        if case.vignette:
            rs.append((case.shape, case.cfgkw, case.req))
    cfgs = [dict(allow_experiments=True, max_filters=8), dict(allow_experiments=True), EXP]
    for shape in [(60, 80, 3), (45, 64, 4), (33, 47, 1), (48, 64, 3), (97, 33, 3), (131, 259, 4)]:
        for rq in REQS:
            if any("vignette" in f for f in rq.get("filters", [])):
                rs += [(shape, kw, rq) for kw in cfgs]
    edge = dict(filters=["rotate=90", "vignette=0.8", "blur=1"])
    rs += [((h, w, c), dict(allow_experiments=True, max_filters=8), edge)
           for (h, w, c) in [(1, 1, 3), (1, 1, 4), (1, 7, 1), (9, 1, 4), (2, 3, 3), (8, 32, 4), (9, 33, 3), (257, 3, 3)]]
    cfg4 = dict(filters=["blur=2.3", "vignette=0.8", "rotate=90"])
    rs += [((3000, 4000, 3), dict(allow_experiments=True), cfg4), ((750, 1000, 3), EXP, cfg4), ((61, 79, 3), EXP, cfg4),
           ((216, 384, 4), EXP, cfg4), ((256, 256, 3), dict(allow_experiments=True), dict(filters=["vignette=0.8"])),
           ((131, 67, 4), dict(allow_experiments=True), dict(filters=["vignette=4,3"])),
           ((256, 256, 4), dict(allow_experiments=True), dict(filters=["vignette=0.5,0.7"]))]
    rs += [(s, EXP, rq) for s, rq in matrix()]
    return rs


def _frames(reqs):
    """{(w, h, cx, cy, maxr, intensity): (op, intensity and radius of its filter)} over the requests' vignette ops."""
    out = {}
    for shape, kw, rq in reqs:
        ops = G.vignette_ops(shape, kw, rq, must_plan=False)
        fs = [f for f in rq.get("filters", []) if f.split("=", 1)[0] == "vignette"]
        for op, f in zip(ops, fs):
            out.setdefault((op["w"], op["h"], op["cx"], op["cy"], float(op["maxr"]), float(op["intensity"])), (op, _vig_args(f)))
    return out


SWEEP = [(1, 1), (2, 1), (1, 2), (3, 3), (4, 5), (17, 16), (64, 64), (65, 63), (320, 240), (321, 241), (640, 480), (1001, 999),
         (1920, 1080), (1081, 1919), (2047, 1537), (3000, 4000), (4000, 3000), (3999, 2999)]


def _check_tables(hostsim, orc, op, args):
    """The oracle's and hostsim's tables against the reference on every exact entry; returns the ambiguous count."""
    import ctypes as C
    w, h, cx, cy = op["w"], op["h"], op["cx"], op["cy"]
    nx, ny = VR.table_dims(w, h, cx, cy)
    mc = VR.classify(op["maxr"], op["intensity"], nx, ny)
    if op["nx"]:                                             # the planner's table: the frame plus the margin, no more, no less
        assert (op["nx"], op["ny"]) == (nx, ny), (op, nx, ny)
    assert (nx * ny <= VR.TABLE_LIMIT) == (op["nx"] > 0), (op, nx * ny)
    o = orc.orc().vignette_mask_table(nx, ny, w, h, *args)
    hs = np.empty((ny, nx), np.float32)
    hostsim.lib.hostsim_vignette_mask_table.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_float]
    hostsim.lib.hostsim_vignette_mask_table(hs.ctypes.data, nx, ny, op["maxr"], op["intensity"])
    ex = ~mc.ambiguous
    for name, t in (("oracle", o), ("hostsim", hs)):
        same = (t == mc.mask) | (np.isnan(t) & np.isnan(mc.mask))
        bad = np.argwhere(ex & ~same)
        assert len(bad) == 0, (name, op, len(bad), [(int(j), int(i), float(t[j, i]), float(mc.mask[j, i])) for j, i in bad[:5]])
        amb_ok = (t == mc.mask) | (t == mc.alt)
        assert amb_ok[mc.ambiguous].all(), (name, op)
    return mc.count


# ---- CPU ---------------------------------------------------------------------------------------------------------------
def test_suite_frames_count_ambiguous_entries_and_tables_match(hostsim, orc):
    frames = _frames(suite_requests())
    assert len(frames) > 100
    total = entries = 0
    for key, (op, args) in sorted(frames.items(), key=lambda kv: -kv[0][0] * kv[0][1]):
        n = _check_tables(hostsim, orc, op, args)
        nx, ny = VR.table_dims(op["w"], op["h"], op["cx"], op["cy"])
        total += n
        entries += nx * ny
        if n or op["w"] * op["h"] >= 1_000_000:
            print(f"vignette frame {op['w']}x{op['h']} maxr={float(op['maxr'])!r} intensity={float(op['intensity'])!r}: "
                  f"{n} ambiguous of {nx * ny} entries")
    print(f"suite: {len(frames)} vignette frames, {entries} table entries, {total} ambiguous")
    # the fixed seeds and shapes of the suite hold no ambiguous entry: every vignette result is compared bit-exactly
    assert total == 0
    assert len(G.UNMAPPED_AMBIGUOUS) == 0


@pytest.mark.parametrize("f", ["vignette=0.8", "vignette=4,3"])
def test_size_sweep_counts_ambiguous_entries_and_tables_match(hostsim, orc, f):
    total = 0
    for (w, h) in SWEEP:
        ops = G.vignette_ops((h, w, 3), EXP, dict(filters=[f]))
        assert len(ops) == 1 and (ops[0]["w"], ops[0]["h"]) == (w, h)
        n = _check_tables(hostsim, orc, ops[0], _vig_args(f))
        total += n
        print(f"{f} {w}x{h}: {n} ambiguous")
    print(f"{f}: {total} ambiguous entries over {len(SWEEP)} frames")


def test_delta_is_the_largest_documented_bound():
    import mpmath
    with mpmath.workdps(60):
        assert VR.DELTA == VR.DELTA_DEV
        assert abs(VR.DELTA * mpmath.mpf(2) ** 52 - mpmath.mpf("9.5")) < mpmath.mpf("1e-12")


def test_decide_at_constructed_boundaries():
    """Values on, within DELTA of and just beyond DELTA of a float rounding boundary: ambiguous with the neighbour as the
    other candidate, or exact with the nearest float."""
    import mpmath
    with mpmath.workdps(60):
        for f in (np.float32(0.7), np.float32(0.25), np.float32(1e-30), np.float32(0.9999999)):
            up = np.nextafter(f, np.float32(2))
            m = (mpmath.mpf(float(f)) + mpmath.mpf(float(up))) / 2
            for k, amb in ((0, True), (mpmath.mpf("0.999"), True), (mpmath.mpf("1.001"), False)):
                for side in (-1, 1):
                    t = m * (1 + side * k * VR.DELTA)
                    g, a, alt = VR.decide(t)
                    assert a == amb, (f, k, side)
                    near = f if (t < m or (t == m and side < 0)) else up
                    if t != m:
                        assert g == near, (f, k, side, g)
                    assert (alt != g) == amb and (not amb or {g, alt} == {f, up}), (f, k, side, g, alt)
    mc = VR.classify_raw(np.array([0.0, 0.5, 1.0, 3.0], np.float32))
    assert mc.mask[0] == 1.0 and mc.count == 0
    with mpmath.workdps(60):
        for x, m in zip((0.5, 1.0, 3.0), mc.mask[1:]):
            assert VR.decide(mpmath.cos(mpmath.mpf(x)) ** 4)[0] == m


def test_table_limit_sides(hostsim):
    """8048^2 takes a table of 4089^2 entries (<= 16M), 8064^2 evaluates each pixel (4097^2 > 16M); cfg4's frame a table."""
    sides = {}
    for n in (8048, 8064):
        ops = G.vignette_ops((n, n, 1), EXP, dict(filters=["vignette=0.8"]))
        assert len(ops) == 1
        sides[n] = (ops[0]["nx"], ops[0]["ny"])
    assert sides[8048] == (4089, 4089) and 4089 * 4089 <= VR.TABLE_LIMIT
    assert sides[8064] == (0, 0) and 4097 * 4097 > VR.TABLE_LIMIT
    op = G.vignette_ops((3000, 4000, 3), dict(allow_experiments=True), dict(filters=["blur=2.3", "vignette=0.8", "rotate=90"]))[0]
    assert (op["w"], op["h"], op["nx"], op["ny"]) == (4000, 3000, 2065, 1565)
    op = G.vignette_ops((40, 50, 3), EXP, dict(filters=["rotate=90", "vignette=0.8"]))[0]
    assert (op["w"], op["h"], op["cx"], op["cy"]) == (40, 50, 20, 25)


def _gray(img):
    """b = g = r = the first channel (alpha kept): the vignette's S is 0 and its V the pixel's value."""
    g = img.copy()
    if g.shape[2] >= 3:
        g[:, :, 1] = g[:, :, 0]
        g[:, :, 2] = g[:, :, 0]
    return g


def gray_values(h, w, c, full):
    """V = 255 everywhere (full) or every value 0..255 spread over the frame."""
    if full:
        return np.full((h, w, c), 255, np.uint8)
    xx, yy = np.arange(w, dtype=np.int32)[None, :], np.arange(h, dtype=np.int32)[:, None]
    v = ((xx * 7 + yy * 13 + (xx * yy) % 5) % 256).astype(np.uint8)
    img = np.repeat(v[:, :, None], c, axis=2)
    if c == 4:
        img[:, :, 3] = 200
    return img


def expected_gray(orc, img, kw, rq):
    """(expected result, ambiguous output pixels) of a request with one vignette followed by orientations only, on a gray
    image: the steps before the vignette by the oracle (they are compared bit-exactly elsewhere), the vignette as
    trunc(V * mask) from the reference mask, the orientations after it by the oracle's flips and rotations."""
    from oracle import oracle as O
    fs = rq["filters"]
    k = [i for i, f in enumerate(fs) if f.split("=", 1)[0] == "vignette"]
    assert len(k) == 1 and all(f.split("=", 1)[0] in G.ORIENT for f in fs[k[0] + 1:]), rq
    k = k[0]
    code, _, v = _oracle(orc, img, dict(rq, filters=fs[:k]), kw)
    assert code == 0, rq
    assert (v[:, :, 1] == v[:, :, 0]).all() and (v[:, :, 2] == v[:, :, 0]).all(), rq
    op = G.vignette_ops(img.shape, kw, rq)[0]
    assert (op["h"], op["w"]) == v.shape[:2], (rq, op, v.shape)
    m, amb = VR.gray_expected(op, v[:, :, 0])
    out = v.copy()
    out[:, :, :3] = m[:, :, None]
    ambi = np.repeat(amb[:, :, None].astype(np.uint8), 3, axis=2)
    for f in fs[k + 1:]:
        _, out = O.apply_filter(out, f, True)
        _, ambi = O.apply_filter(ambi, f, True)
    return out, ambi[:, :, 0] > 0


def assert_gray(out, exp, amb, label):
    """Exact but at ambiguous pixels, which may differ by 1."""
    assert out.shape == exp.shape, (label, out.shape, exp.shape)
    d = np.abs(out.astype(np.int16) - exp.astype(np.int16))
    assert d.max(initial=0) <= 1 and d[~amb].max(initial=0) == 0, (label, int(d.max()), int((d[~amb] > 0).sum()), d.size)
    if amb.any():
        G.VIGNETTE_ALLOWANCE_USED.append((repr(label), int(amb.sum()), int((d > 0).sum())))


def test_hostsim_gray_frames_against_the_reference_mask(hostsim, orc):
    n = 0
    for full in (True, False):
        for (h, w, c), rq in matrix():
            img = gray_values(h, w, c, full)
            code, _, out = hostsim.run(img, api.Config(**EXP), **rq)
            assert code == 0, rq
            assert_gray(out, *expected_gray(orc, img, EXP, rq), (full, (h, w), rq))
            n += 1
    for case in kernel_family_cases():
        h, w, c = case.shape
        if h * w > 300_000:
            continue
        img = _gray(case.image())
        code, _, out = hostsim.run(img, api.Config(**case.cfgkw), **case.req)
        assert code == 0
        assert_gray(out, *expected_gray(orc, img, case.cfgkw, case.req), case.name)
        n += 1
    assert n > 150


def test_hostsim_vignette_requests_of_the_planner_matrix_are_exact(hostsim, orc):
    """hostsim against the oracle on test_planner_host's vignette requests: no ambiguous entry, so bit-exact."""
    n = 0
    for shape in [(60, 80, 3), (45, 64, 4), (33, 47, 1), (48, 64, 3)]:
        img = smooth_image(shape[0] + shape[1], *shape)
        for rq in REQS:
            if not any("vignette" in f for f in rq.get("filters", [])):
                continue
            code, _, out = hostsim.run(img, api.Config(**EXP), **rq)
            c2, _, ref = _oracle(orc, img, rq, EXP)
            assert code == c2
            if code:
                continue
            allowed, n_amb = G.vignette_allowance(img.shape, EXP, rq, out.shape)
            assert allowed is None and n_amb == 0, rq
            assert np.array_equal(out, ref), rq
            n += 1
    assert n >= 12


# ---- GPU ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_gray_frames_against_the_reference_mask(gpu, orc):
    from test_gpu_parity import _gpu_run
    from test_kernel_branches import run_case_gpu
    n = 0
    for full in (True, False):
        for (h, w, c), rq in matrix():
            img = gray_values(h, w, c, full)
            code, _, out = _gpu_run(gpu, img, EXP, rq)
            assert code == 0, (rq, gpu.last_error())
            assert_gray(out, *expected_gray(orc, img, EXP, rq), (full, (h, w), rq))
            n += 1
    for case in kernel_family_cases():
        img = _gray(case.image())
        assert_gray(run_case_gpu(gpu, case, img), *expected_gray(orc, img, case.cfgkw, case.req), case.name)
        n += 1
    assert n > 150


@pytest.mark.gpu
def test_gpu_colour_frames_against_the_oracle(gpu, orc):
    from test_gpu_parity import _gpu_run
    from test_kernel_branches import run_case_gpu
    for k, ((h, w, c), rq) in enumerate(matrix()):
        for cc in (3, 4):
            img = smooth_image(k, h, w, cc) if k % 2 else rnd_image(k, h, w, cc)
            code, _, out = _gpu_run(gpu, img, EXP, rq)
            c2, _, ref = _oracle(orc, img, rq, EXP)
            assert code == c2 == 0, (rq, code, c2)
            G.assert_vignette_exact(out, ref, img.shape, EXP, rq, ((h, w, cc), rq))
    for case in kernel_family_cases():
        img = case.image()
        ref = _oracle(orc, img, case.req, case.cfgkw)[2]
        G.assert_vignette_exact(run_case_gpu(gpu, case, img), ref, case.shape, case.cfgkw, case.req, case.name)


@pytest.mark.gpu
def test_gpu_table_and_per_pixel_sides_of_the_limit(gpu):
    """8048^2 (mask table) and 8064^2 (CUDA's double cos per pixel in the pass kernel), 1-channel sources holding every value:
    both exact against the reference mask, and the table costs exactly one more launch on first use."""
    from test_gpu_parity import _gpu_run
    rq = dict(filters=["vignette=0.8"])
    launches = {}
    for n in (8048, 8064):
        img = gray_values(n, n, 1, False)
        op = G.vignette_ops(img.shape, EXP, rq)[0]
        assert (op["nx"] > 0) == (n == 8048)
        before = gpu.launch_count()
        code, _, out = _gpu_run(gpu, img, EXP, rq)
        launches[n] = gpu.launch_count() - before
        assert code == 0, gpu.last_error()
        m, amb = VR.gray_expected(op, img[:, :, 0])
        exp = np.repeat(m[:, :, None], out.shape[2], axis=2)
        del m
        assert_gray(out, exp, amb, f"{n}x{n}")
        del out, exp, img
    assert launches[8048] == launches[8064] + 1, launches


@pytest.mark.gpu
def test_zz_report_allowance_use():
    """Runs after this module's GPU tests: prints how many comparisons used the ambiguous-pixel allowance."""
    used = G.VIGNETTE_ALLOWANCE_USED
    print(f"vignette allowance used by {len(used)} comparisons, {sum(u[2] for u in used)} bytes differed there: {used[:10]}")
