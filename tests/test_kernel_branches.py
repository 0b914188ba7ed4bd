"""Every kernel branch the planner can select, against the oracle (tests/kernel_cases.py holds the branch table and the
cases). On the CPU: each case lands on the branch it names, the cases cover the whole table but an argued list of
unreachable branches, the footprint-limit pairs fall on either side of their limit, and hostsim's walk of the small cases
equals the oracle. On the GPU: each case bit-exact through imp_gpu_run_host, all of them in one device batch, the device
buffer layouts imp_gpu_run_device / imp_gpu_batch_add accept (nothing outside a result row's w*c bytes may change), and
the whole list over the bounds-checking debug build."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import golden_util as G
import kernel_cases as K
from ngx_http_imgproc_b200 import api
from test_planner_host import _oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CASES = K.all_cases()
CANARY = 0xA5


# ---- CPU -----------------------------------------------------------------------------------------------------------
def _landing(hostsim, case):
    """The pass of the case's plan that is on the case's branch (with the fields it pins), or None."""
    for b in K.plan_branches(hostsim, case):
        if K.branch_key(b) == case.branch and all(b[k] == v for k, v in case.expect.items()):
            return b
    return None


def test_case_names_are_unique():
    names = [c.name for c in CASES]
    assert len(names) == len(set(names))


def test_every_case_lands_on_its_branch(hostsim):
    missed = []
    for case in CASES:
        if _landing(hostsim, case) is None:
            missed.append((case.name, case.branch, case.expect, [(K.branch_key(b), b) for b in K.plan_branches(hostsim, case)]))
    assert not missed, missed[:5]


def test_cases_cover_the_branch_table(hostsim):
    table = K.table()
    assert set(K.UNREACHABLE) <= table and all(K.UNREACHABLE.values())
    reached = set()
    for case in CASES:
        reached |= {K.branch_key(b) for b in K.plan_branches(hostsim, case)}
    assert reached <= table, sorted(reached - table)
    assert not reached & set(K.UNREACHABLE), sorted(reached & set(K.UNREACHABLE))
    missing = table - reached - set(K.UNREACHABLE)
    assert not missing, sorted(missing)
    # the dispatch switches of the strip kernel, case by case
    for mode in ("area_frac", "area_int"):
        for sc in (1, 3, 4):
            for fl in (0, 1, 2):
                assert {n for n in range(1, 13) if ("strip", mode, n, sc, fl) in reached} == set(range(1, 13)), (mode, sc, fl)


@pytest.mark.parametrize("limit", [name for name, _, _ in K.limit_pairs()])
def test_limit_pairs_straddle_their_limit(hostsim, limit):
    """The inside case keeps its tile kernel; the outside case takes the next smaller tile (same kernel, smaller edge) or
    the pass's fallback, and is otherwise the same request on a source a step larger (or with one table more)."""
    _, inside, outside = [p for p in K.limit_pairs() if p[0] == limit][0]
    bi, bo = _landing(hostsim, inside), _landing(hostsim, outside)
    assert bi is not None and bo is not None, (limit, K.plan_branches(hostsim, inside), K.plan_branches(hostsim, outside))
    assert bi["kernel"] not in (K.DIRECT, K.CUBIC_RUN, K.BLUR_GENERIC) and bi["smem_bytes"] <= K.SMEM_OPTIN, bi
    if bo["kernel"] == bi["kernel"]:
        assert bo["kernel"] == K.STRIP or 0 < bo["gt"] < bi["gt"], (limit, bi, bo)    # LINEAR 1.25: gather tile -> strip
        assert bo["kernel"] != K.STRIP or bi["kernel"] == K.STRIP and bi["kind"] == bo["kind"] == K.G_LINEAR
    else:
        kind = K.KIND[bo["kind"]]
        assert bo["kernel"] == {"cubic": K.CUBIC_RUN, "blur": K.BLUR_GENERIC}.get(kind, K.DIRECT) or \
            (bi["kernel"] == K.GATHER_TILE and bo["kernel"] == K.STRIP), (limit, bo)


def test_integer_strip_consumer_stays_within_its_switch(hostsim):
    """The integer consumer is instantiated with NT = nx for nx 1..12 and `default: 12`: a wider box must never reach it.
    max_xtaps <= 12 keeps every nx > 12 (and every fractional pass with more than 12 taps) off the strip kernel."""
    for n in (13, 14, 16, 24):
        for sc in (1, 3, 4):
            case = K.Case("x", (K.SH, K.SW * n, sc), K.BASE_KW, dict(K.INT12), ("direct", "area_int", sc))
            (b,) = K.plan_branches(hostsim, case)
            assert b["kind"] == K.G_AREA_INT and b["nx"] == n and b["kernel"] == K.DIRECT, b


def test_hostsim_matches_oracle_on_the_small_cases(hostsim, orc):
    n = 0
    for case in CASES:
        h, w, c = case.shape
        if h * w > 300_000:
            continue
        img = case.image()
        code, _, out = hostsim.run(img, api.Config(**case.cfgkw), **case.req)
        c2, _, ref = _oracle(orc, img, case.req, case.cfgkw)
        assert code == c2 == 0, case.name
        _assert_same(out, ref, case)
        n += 1
    assert n > 250


def _assert_same(out, ref, case):
    assert out.shape == ref.shape, (case.name, out.shape, ref.shape)
    d = np.abs(out.astype(int) - ref.astype(int))
    if case.vignette:
        G.assert_vignette_exact(out, ref, case.shape, case.cfgkw, case.req, case.name)
    else:
        assert d.max() == 0, (case.name, int(d.max()), int((d > 0).sum()), d.size)


# ---- device buffers inside canaries ----------------------------------------------------------------------------------
class DevRows:
    """h rows of row_bytes at (base + off, pitch) inside one device allocation filled with CANARY: 64 bytes before, the
    pitch padding between the rows and 64 bytes after must still hold it after a run."""

    LEAD = 64

    def __init__(self, gpu, h, row_bytes, pitch, off, rows=None):
        self.gpu, self.h, self.row, self.pitch, self.off = gpu, h, row_bytes, pitch, off
        self.total = self.LEAD + off + pitch * h + 64
        d, p = C.c_void_p(), C.c_int()
        gpu.check(gpu.lib.imp_gpu_malloc_pitch(C.byref(d), C.byref(p), self.total, 1))
        self.base = d.value
        self.ptr = self.base + self.LEAD + off
        self.fill()
        if rows is not None:
            rows = np.ascontiguousarray(rows)
            gpu.check(gpu.lib.imp_gpu_upload_2d(self.ptr, pitch, rows.ctypes.data, rows.strides[0], row_bytes, h, None))
        gpu.check(gpu.lib.imp_gpu_sync(None))

    def fill(self):
        """Every byte of the allocation back to CANARY."""
        fill = np.full(self.total, CANARY, np.uint8)
        self.gpu.check(self.gpu.lib.imp_gpu_upload_2d(self.base, self.total, fill.ctypes.data, self.total, self.total, 1, None))
        self.gpu.check(self.gpu.lib.imp_gpu_sync(None))

    def read(self, shape):
        """(pixels as `shape`, whether every byte outside the rows' spans still holds the canary)."""
        raw = np.empty(self.total, np.uint8)
        self.gpu.check(self.gpu.lib.imp_gpu_download_2d(raw.ctypes.data, self.total, self.base, self.total, self.total, 1, None))
        self.gpu.check(self.gpu.lib.imp_gpu_sync(None))
        inside = np.zeros(self.total, bool)
        first = self.LEAD + self.off
        for y in range(self.h):
            inside[first + y * self.pitch: first + y * self.pitch + self.row] = True
        px = np.stack([raw[first + y * self.pitch: first + y * self.pitch + self.row] for y in range(self.h)]).reshape(shape)
        return px, bool((raw[~inside] == CANARY).all())

    def free(self):
        self.gpu.lib.imp_gpu_free(self.base)


def _src_pitch(row, pad):
    return row + pad if pad else (row + 15) & ~15


def run_case_gpu(gpu, case, img):
    """The case on the GPU: through imp_gpu_run_host, or, for a padded source (pitch % 16 != 0: the fallback kernels),
    through imp_gpu_run_device on device rows src_pad bytes longer than a source row."""
    h, w, c = case.shape
    p = gpu.plan(w, h, c, api.Config(**case.cfgkw), **case.req)
    try:
        if not case.src_pad:
            return p.run_host(img)
        src = DevRows(gpu, h, w * c, w * c + case.src_pad, 0, img)
        dst = DevRows(gpu, p.out_h, p.out_w * p.out_c, (p.out_w * p.out_c + 15) & ~15, 0)
        p.run_device(src.ptr, src.pitch, dst.ptr, dst.pitch)
        out, clean = dst.read((p.out_h, p.out_w, p.out_c))
        src.free(); dst.free()
        assert clean, case.name
        return out
    finally:
        p.close()


@pytest.fixture(scope="module")
def refs(orc):
    cache = {}

    def get(case):
        if case.name not in cache:
            code, _, ref = _oracle(orc, case.image(), case.req, case.cfgkw)
            assert code == 0, case.name
            cache[case.name] = ref
        return cache[case.name]
    return get


# ---- GPU -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_every_case_matches_the_oracle(gpu, refs):
    for case in CASES:
        _assert_same(run_case_gpu(gpu, case, case.image()), refs(case), case)


@pytest.mark.gpu
def test_all_cases_in_one_device_batch(gpu, refs):
    """Every case as one job of ONE imp_gpu_batch: jobs are grouped by (kind, sc, kernel, param, flavour, occupancy class),
    so the batch holds many groups, and a group's launch takes the largest footprint of its jobs."""
    batch = api.Batch(gpu)
    jobs = []
    try:
        for case in CASES:
            h, w, c = case.shape
            img = case.image()
            p = gpu.plan(w, h, c, api.Config(**case.cfgkw), **case.req)
            src = DevRows(gpu, h, w * c, _src_pitch(w * c, case.src_pad), 0, img)
            dst = DevRows(gpu, p.out_h, p.out_w * p.out_c, (p.out_w * p.out_c + 15) & ~15, 0)
            batch.add(p, src.ptr, src.pitch, dst.ptr, dst.pitch)
            jobs.append((case, p, src, dst))
        # The first launch also brings every plan to the device, which builds one vignette mask table per vignette op (a
        # kernel of its own, counted by imp_gpu_launch_count); a second launch of the same batch runs only its groups.
        tables = sum(1 for case in CASES if case.vignette)
        for run in range(2):
            for _, _, _, dst in jobs:
                dst.fill()                                 # the second run is checked on its own writes
            before = gpu.launch_count()
            batch.launch()
            gpu.check(gpu.lib.imp_gpu_sync(None))
            launches = gpu.launch_count() - before
            per_run = batch.launches_per_run
            assert launches == per_run + (tables if run == 0 else 0) and per_run < len(CASES) // 2, (run, launches, per_run, tables)
            for case, p, src, dst in jobs:
                out, clean = dst.read((p.out_h, p.out_w, p.out_c))
                assert clean, (run, case.name)
                _assert_same(out, refs(case), case)
    finally:
        for _, p, src, dst in jobs:
            src.free(); dst.free(); p.close()
        batch.close()


def layout_cases():
    """One request per kernel family x source channels x result channels (FI24 / FI32 packing included). Each reads a
    crop window whose first byte is 16-byte aligned when the image base is 4 bytes past an aligned address, so that
    layout still takes the tile kernel."""
    fams = {"strip_frac": (dict(resize="45,37"), (83, 101)), "strip_int": (dict(resize="45,37"), (74, 135)),
            "strip_linear": (dict(resize="45,37", interp=1), (83, 101)), "gather_copy": (dict(filters=["rotate=90"]), (37, 45)),
            "gather_nn": (dict(resize="91,67,up", simple=True), (37, 45)), "gather_linear": (dict(resize="91,67,up", interp=1), (37, 45)),
            "cubic": (dict(resize="91,67,up", filters=["flip=10"]), (37, 45)), "blur": (dict(filters=["blur=1.5", "rotate=270"]), (53, 61))}
    out = []
    for fam, (rq, (wh, ww)) in fams.items():
        for sc in (1, 3, 4):
            x0 = {1: 12, 3: 4, 4: 3}[sc]                   # (4 + x0 * sc) % 16 == 0
            for pack in ((0, 24) if sc == 4 else (0, 32)):
                r = dict(rq, crop=f"{ww}px,{wh}px,{x0}px,2px", pack=pack)
                out.append(K.Case(f"layout_{fam}_c{sc}_p{pack}", (wh + 5, ww + x0 + 3, sc), K.BASE_KW, r, None))
    return out


def _layouts(case, out_c):
    """(source layouts, destination layouts) as (name, pitch function of the row, base offset)."""
    srcs = [("aligned", lambda r: (r + 15) & ~15, 0), ("base+4", lambda r: (r + 15) & ~15, 4),
            ("pitch%16", lambda r: r + (4 if (r + 4) % 16 else 8), 0)]
    dsts = [("aligned", lambda r: (r + 15) & ~15, 0), ("pitch+4,base+4", lambda r: r + 4, 4)]
    if out_c == 3:
        dsts.append(("pitch+1,base+1", lambda r: r + 1, 1))
    return srcs, dsts


@pytest.mark.gpu
def test_device_layouts_match_the_oracle_and_write_only_the_rows(gpu, refs):
    """imp_gpu_run_device and imp_gpu_batch_add over every layout the device-buffer contract (include/imp_gpu.h) allows:
    destinations 16-byte aligned, 4 bytes off (pitch row + 4), and for 3-channel results 1 byte off (pitch row + 1);
    sources aligned, 4 bytes off with a 16-byte aligned window (tile kernels), and with a pitch that is not a multiple of 16
    (the fallback kernels). The pixels equal the oracle's; the bytes around and between the rows keep the canary."""
    batch = api.Batch(gpu)
    plans, bufs, pending = [], [], []
    try:
        for case in layout_cases():
            h, w, c = case.shape
            ref = refs(case)
            p = gpu.plan(w, h, c, api.Config(**case.cfgkw), **case.req)
            plans.append(p)
            srcs, dsts = _layouts(case, p.out_c)
            row = p.out_w * p.out_c
            for sname, spitch, soff in srcs:
                src = DevRows(gpu, h, w * c, spitch(w * c), soff, case.image())
                bufs.append(src)
                for dname, dpitch, doff in dsts:
                    tag = f"{case.name} src {sname} dst {dname}"
                    dst = DevRows(gpu, p.out_h, row, dpitch(row), doff)
                    bufs.append(dst)
                    p.run_device(src.ptr, src.pitch, dst.ptr, dst.pitch)
                    out, clean = dst.read(ref.shape)
                    assert clean, ("imp_gpu_run_device wrote outside the rows", tag)
                    _assert_same(out, ref, K.Case(tag, case.shape, case.cfgkw, case.req, None))
                    dst = DevRows(gpu, p.out_h, row, dpitch(row), doff)
                    bufs.append(dst)
                    batch.add(p, src.ptr, src.pitch, dst.ptr, dst.pitch)
                    pending.append((dst, ref, case, tag))
        batch.launch()
        gpu.check(gpu.lib.imp_gpu_sync(None))
        for dst, ref, case, tag in pending:
            out, clean = dst.read(ref.shape)
            assert clean, ("the batch wrote outside the rows", tag)
            _assert_same(out, ref, K.Case(tag, case.shape, case.cfgkw, case.req, None))
    finally:
        for b in bufs:
            b.free()
        for p in plans:
            p.close()
        batch.close()
    n = len(pending)
    assert n == 8 * 6 * 3 * 2 + 8 * 3 * 3, n       # 3-channel results: one destination layout more


@pytest.mark.gpu
def test_device_layouts_outside_the_contract_are_refused(gpu):
    """4-channel rows must be 4-byte addressable: check_device_job refuses the rest before any work."""
    case = [c for c in layout_cases() if c.name == "layout_strip_frac_c4_p0"][0]
    h, w, c = case.shape
    p = gpu.plan(w, h, c, api.Config(**case.cfgkw), **case.req)
    src = DevRows(gpu, h, w * c, (w * c + 15) & ~15, 0, case.image())
    row = p.out_w * 4
    dst = DevRows(gpu, p.out_h, row, row + 4, 0)
    batch = api.Batch(gpu)
    try:
        for sp, soff, dp, doff in [((w * c + 15) & ~15, 0, row + 2, 0), ((w * c + 15) & ~15, 0, row + 4, 2),
                                   (w * c + 2, 0, row + 4, 0), ((w * c + 15) & ~15, 1, row + 4, 0), ((w * c + 15) & ~15, 0, row - 4, 0)]:
            assert gpu.lib.imp_gpu_run_device(p.h, src.ptr + soff, sp, dst.ptr + doff, dp, None) == 50
            assert gpu.lib.imp_gpu_batch_add(batch.h, p.h, src.ptr + soff, sp, dst.ptr + doff, dp) == 50
        gpu.check(gpu.lib.imp_gpu_sync(None))
        assert gpu.lib.imp_gpu_batch_size(batch.h) == 0
        _, clean = dst.read((p.out_h, p.out_w, 4))
        assert clean
    finally:
        src.free(); dst.free(); p.close(); batch.close()


@pytest.mark.gpu
def test_every_case_over_the_debug_build(orc):
    """The whole case list over libimp_gpu_dbg.so (-DIMP_DEBUG_BOUNDS: every staged-tile, lookup, out-stage and destination
    address the tile kernels form is checked) in a child process: no assertion fires, the outputs equal the oracle's."""
    dbg = os.path.join(ROOT, "ngx_http_imgproc_b200", "libimp_gpu_dbg.so")
    assert os.path.exists(dbg), "debug library not built (python -m ngx_http_imgproc_b200.build --debug)"
    code = r"""
import sys, ctypes as C
sys.path.insert(0, "."); sys.path.insert(0, "tests")
import ngx_http_imgproc_b200 as M
from oracle import oracle as O
import kernel_cases as K
from test_planner_host import _oracle
from test_kernel_branches import run_case_gpu, _assert_same
L = M.library(); L.init(0)
L.lib.imp_gpu_debug_flags.restype = C.c_uint
n = 0
for case in K.all_cases():
    img = case.image()
    code, _, ref = _oracle(O, img, case.req, case.cfgkw)
    assert code == 0, case.name
    _assert_same(run_case_gpu(L, case, img), ref, case)
    n += 1
flags = L.lib.imp_gpu_debug_flags()
print("BOUNDS", n, hex(flags))
assert flags == 0, hex(flags)
"""
    env = dict(os.environ, IMP_GPU_LIB=dbg)
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "BOUNDS" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]
    assert int(r.stdout.split("BOUNDS")[1].split()[0]) == len(CASES)
