"""Many GIF albums in one call (imp_gpu_gif_albums_run_host).

CPU: where the album list is cut into rounds (imp_gif_round_bounds, restated here: consecutive albums while the sum of their
canvas bytes a256(a16(4 cw) ch n_pages) stays within 256 MB, an album above it alone), and the expansion of one packed
multi-album round by the code the kernel compiles (imp_gif_expand_thread over imp_gif_pack_page's block, on the CPU), each
album against the oracle's LoadGIF restatement of that album alone.

GPU: a mixed batch bit-exact against the oracle chain and against one gif_album call per album, whatever n_streams and the
album order; one expansion launch per round; several rounds; nothing written when one album is bad; the debug build."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from ngx_http_imgproc_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MB = 1 << 20
BUDGET = 256 * MB
NN_SEPIA = dict(simple=True, filters=["modulate=0,0,100", "colorize=704214,0.6"])


def a16(v):
    return (v + 15) & ~15


def a256(v):
    return (v + 255) & ~255


def canvas_bytes(cw, ch, n):
    return a256(a16(4 * cw) * ch * n)


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("gifshim") / "libgif_shim.so")
    cuda_inc = os.environ.get("CUDA_HOME", "/usr/local/cuda") + "/include"
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-w", "-I" + cuda_inc, "-o", so,
                    os.path.join(ROOT, "tests", "hostsim", "gif_shim.cpp"),
                    os.path.join(ROOT, "tests", "hostsim", "transfer_shim.cpp"),
                    os.path.join(ROOT, "ngx_http_imgproc_b200", "csrc", "imp_transfer.cpp")], check=True)
    lib = C.CDLL(so)
    lib.shim_gif_round_bounds.argtypes = [C.c_int, C.c_void_p, C.c_void_p]
    lib.shim_gif_expand.argtypes = [C.c_int, C.c_void_p, C.c_void_p]
    lib.shim_gif_expand.restype = C.c_longlong
    lib.shim_bounds.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_void_p]
    lib.shim_plan.restype = C.c_void_p
    lib.shim_plan.argtypes = [C.c_int] * 10
    lib.shim_plan_free.argtypes = [C.c_void_p]
    return lib


def round_bounds(shim, geoms):
    """geoms: (cw, ch, n_pages) per album; only the geometry is read."""
    arr = (api.CGifAlbum * max(len(geoms), 1))(*[api.CGifAlbum(None, n, cw, ch, 1, None, None, None) for cw, ch, n in geoms])
    out = (C.c_int * (len(geoms) + 2))()
    k = shim.shim_gif_round_bounds(len(geoms), arr, out)
    return list(out[:k])


def restated_bounds(geoms):
    b, i = [0], 0
    while i < len(geoms):
        e, tot = i, 0
        while e < len(geoms):
            need = canvas_bytes(*geoms[e])
            if e > i and tot + need > BUDGET:
                break
            tot += need
            e += 1
        b.append(e)
        i = e
    return b


def test_round_bounds_cover_consecutive_within_budget(shim):
    rng = np.random.default_rng(3)
    for trial in range(40):
        geoms = [(int(rng.integers(1, 2000)), int(rng.integers(1, 1200)), int(rng.integers(1, 60))) for _ in range(int(rng.integers(1, 40)))]
        b = round_bounds(shim, geoms)
        assert b == restated_bounds(geoms), trial
        assert b[0] == 0 and b[-1] == len(geoms) and all(x < y for x, y in zip(b, b[1:]))
        for r0, r1 in zip(b, b[1:]):
            tot = sum(canvas_bytes(*g) for g in geoms[r0:r1])
            assert r1 - r0 == 1 or tot <= BUDGET
            if r1 < len(geoms):                                   # greedy: the next album would not have fitted
                assert tot + canvas_bytes(*geoms[r1]) > BUDGET


def test_round_bounds_budget_edge(shim):
    quarter = (1024, 1024, 16)                                    # 4 MB per page, 64 MB per album
    assert canvas_bytes(*quarter) * 4 == BUDGET
    assert round_bounds(shim, [quarter] * 4) == [0, 4]            # exactly the budget: one round
    assert round_bounds(shim, [quarter] * 4 + [(1, 1, 1)]) == [0, 4, 5]
    assert round_bounds(shim, [quarter] * 8) == [0, 4, 8]


def test_round_bounds_oversize_album_alone(shim):
    big = (1024, 1024, 65)                                        # 260 MB: above the budget
    small = (160, 120, 24)
    assert canvas_bytes(*big) > BUDGET
    assert round_bounds(shim, [small, big, small]) == [0, 1, 2, 3]
    assert round_bounds(shim, [big]) == [0, 1]
    assert round_bounds(shim, [big, big]) == [0, 1, 2]


def test_round_bounds_count_replay_only_pages(shim):
    # a `page=63` request: 63 replay-only pages and one with a plan; its canvases are all written, so all 64 count
    page_req = (1024, 1024, 64)
    assert round_bounds(shim, [page_req, (1, 1, 1)]) == [0, 1, 2]
    assert round_bounds(shim, [(1024, 1024, 1), (1, 1, 1)]) == [0, 2]


def test_round_bounds_empty(shim):
    assert round_bounds(shim, []) == [0]


def _pages(rng, cw, ch, n, padded):
    """Random pages; padded: FreeImage's 4-byte scanline padding, so the x == left+w over-read meets real pad bytes."""
    out = []
    for f in range(n):
        w = cw if f == 0 else int(rng.integers(1, cw + 1)); h = ch if f == 0 else int(rng.integers(1, ch + 1))
        pitch = (w + 3) & ~3 if padded else w
        out.append(dict(indices=np.ascontiguousarray(rng.integers(0, 16, (h, pitch), dtype=np.uint8)), width=w,
                        left=0 if f == 0 else int(rng.integers(0, cw - w + 1)), top=0 if f == 0 else int(rng.integers(0, ch - h + 1)),
                        dispose=int(rng.integers(0, 4)), key=int(rng.choice([-1, 0, 3, 7])), palette=rng.integers(0, 256, (256, 4), dtype=np.uint8)))
    return out


def test_hostsim_multi_album_round_matches_oracle(shim, orc):
    """One packed round of albums of different sizes (1x1, 160x120, 131x77 whose last block is part-filled) and both
    `destructive` values, expanded by imp_gif_expand_thread over the whole grid: each album equals the oracle on it alone."""
    rng = np.random.default_rng(17)
    o = orc.orc()
    specs = [(1, 1, 3, True), (160, 120, 5, False), (131, 77, 6, True), (131, 77, 4, False), (1, 1, 2, False), (160, 120, 3, True), (7, 300, 4, True)]
    albums = [(_pages(rng, cw, ch, n, padded=k % 2 == 0), cw, ch, d) for k, (cw, ch, n, d) in enumerate(specs)]
    keep, entries = [], []
    for pages, cw, ch, d in albums:
        arr, k = api.Library.gif_pages(pages)
        keep += [arr, k]
        entries.append(api.CGifAlbum(C.addressof(arr), len(pages), cw, ch, 1 if d else 0, None, None, None))
    outs = [np.zeros((len(p), ch, cw, 4), np.uint8) for p, cw, ch, _ in albums]
    tab = (api.CGifAlbum * len(entries))(*entries)
    ptrs = (C.c_void_p * len(outs))(*[x.ctypes.data for x in outs])
    blocks = shim.shim_gif_expand(len(entries), tab, ptrs)
    assert blocks == sum((cw * ch + 255) // 256 for cw, ch, _, _ in specs)
    for (pages, cw, ch, d), got in zip(albums, outs):
        want = o.gif_expand(pages, cw, ch, d)
        for f, w in enumerate(want):
            assert np.array_equal(got[f], w), (cw, ch, d, f)


# ---- on the GPU -------------------------------------------------------------------------------------------------------
def _plan(gpu, cw, ch, rq):
    code, _, plan = gpu.try_plan(cw, ch, 4, api.Config(), **rq)
    assert code == 0, rq
    return plan


def _mixed(gpu, rng):
    """~12 albums: canvas sizes, page counts 1, 2 and 40, both `destructive` values, transparency keys including -1, and
    plans NN simple, cubic enlarge, crop + filters + rotate=90, the empty plan, and a page=N album."""
    specs = [((48, 27, 2), dict(resize="96,54", simple=True), True),
             ((131, 77, 40), dict(crop="100px,60px,c,c", resize="50", filters=["modulate=0,0,100", "colorize=704214,0.6", "rotate=90"]), False),
             ((64, 64, 40), dict(resize="128,128,up", filters=["gamma=1.3"]), True),
             ((33, 21, 1), dict(), True),
             ((1, 1, 2), dict(), False),
             ((90, 52, 7), "page", True),
             ((160, 120, 24), dict(resize="80,60", **NN_SEPIA), True),
             ((320, 240, 2), dict(resize="160,120", **NN_SEPIA), False),
             ((131, 77, 1), dict(resize="262,154,up"), False),
             ((40, 300, 40), dict(resize="20,150", simple=True, filters=["rotate=90"]), True),
             ((200, 30, 2), dict(crop="150px,20px,r,b"), True),
             ((90, 52, 7), dict(resize="45,26", simple=True, filters=["flip=10"]), False)]
    albums, plans, rqs = [], [], []
    for (cw, ch, n), rq, d in specs:
        pages = _pages(rng, cw, ch, n, padded=bool(rng.integers(0, 2)))
        pages[0]["key"] = -1 if len(albums) % 3 == 0 else pages[0]["key"]
        if rq == "page":
            rq = dict(resize="45,26", simple=True)
            p = _plan(gpu, cw, ch, rq)
            per = [None] * (n - 1) + [p]
        else:
            p = _plan(gpu, cw, ch, rq)
            per = [p] * n
        plans.append(p)
        rqs.append(rq)
        albums.append((pages, cw, ch, d, per))
    return albums, plans, rqs


def _copy(outs):
    return [[None if o is None else o.copy() for o in a] for a in outs]


def _assert_albums_equal(a, b, what):
    assert len(a) == len(b)
    for i, (x, y) in enumerate(zip(a, b)):
        assert len(x) == len(y)
        for f, (p, q) in enumerate(zip(x, y)):
            assert (p is None) == (q is None), (what, i, f)
            if p is not None:
                assert p.shape == q.shape and np.array_equal(p, q), (what, i, f)


@pytest.mark.gpu
def test_mixed_albums_bit_exact(gpu, orc):
    from test_planner_host import _oracle
    rng = np.random.default_rng(41)
    o = orc.orc()
    albums, plans, rqs = _mixed(gpu, rng)
    try:
        got = _copy(gpu.gif_albums(albums, n_streams=4))
        for (pages, cw, ch, d, per), rq, outs in zip(albums, rqs, got):
            alone = gpu.gif_album(pages, cw, ch, d, per)
            canvases = o.gif_expand(pages, cw, ch, d)
            for f, (g, a) in enumerate(zip(outs, alone)):
                if per[f] is None:
                    assert g is None and a is None
                    continue
                assert np.array_equal(g, a), (cw, ch, f)
                code, _, ref = _oracle(orc, canvases[f], rq, {})
                assert code == 0 and g.shape == ref.shape and np.array_equal(g, ref), (cw, ch, rq, f)
        _assert_albums_equal(_copy(gpu.gif_albums(albums, n_streams=1)), got, "n_streams=1")
        rev = _copy(gpu.gif_albums(albums[::-1], n_streams=4))[::-1]
        _assert_albums_equal(rev, got, "reversed")
    finally:
        for p in plans:
            p.close()


def _chunks(shim, plan, n_jobs, n_streams):
    ps = [shim.shim_plan(*plan.src, *plan.window, plan.out_w, plan.out_h, plan.out_c) for _ in range(n_jobs)]
    P = (C.c_void_p * n_jobs)(*ps)
    out = (C.c_int * (n_jobs + 2))()
    k = shim.shim_bounds(n_jobs, P, n_streams, out)
    for p in ps:
        shim.shim_plan_free(p)
    return k - 1


@pytest.mark.gpu
def test_one_expansion_launch_per_round(gpu, shim):
    """k thumbnail albums that fit one round: exactly one expansion launch plus one grouped launch per chunk and pass,
    fewer than k single calls take."""
    rng = np.random.default_rng(43)
    k, cw, ch, n = 16, 160, 120, 6
    plan = _plan(gpu, cw, ch, dict(resize="80,60", **NN_SEPIA))
    try:
        albums = [(_pages(rng, cw, ch, n, padded=False), cw, ch, True, plan) for _ in range(k)]
        job = api.GifAlbumsJob(gpu, albums)
        job.run(gpu)                                               # warm: the plan's upload, lanes, buffers
        before = gpu.launch_count()
        job.run(gpu)
        launches = gpu.launch_count() - before
        chunks = _chunks(shim, plan, k * n, 4)
        assert launches - 1 == chunks * plan.passes, (launches, chunks, plan.passes)
        singles = [api.GifAlbumJob(gpu, *a) for a in albums]
        for s in singles:
            s.run(gpu)
        before = gpu.launch_count()
        for s in singles:
            s.run(gpu)
        assert launches < gpu.launch_count() - before
    finally:
        plan.close()


@pytest.mark.gpu
def test_several_rounds(gpu, shim):
    """Albums whose canvases exceed the budget together, and one above it alone: bit-exact against one call per album,
    and one expansion launch per round of imp_gif_round_bounds (counted with replay-only albums, which launch nothing else)."""
    rng = np.random.default_rng(47)
    geoms = [(640, 480, 40)] * 3 + [(1100, 1000, 62)] + [(640, 480, 40)] * 3 + [(96, 64, 3)]
    assert canvas_bytes(1100, 1000, 62) > BUDGET
    plans = {(cw, ch): _plan(gpu, cw, ch, dict(resize=f"{cw // 8},{ch // 8}", **NN_SEPIA)) for cw, ch, _ in geoms}
    try:
        pages = [_pages(rng, cw, ch, n, padded=False) for cw, ch, n in geoms]
        albums = [(p, cw, ch, i % 2 == 0, plans[(cw, ch)]) for i, (p, (cw, ch, n)) in enumerate(zip(pages, geoms))]
        got = _copy(gpu.gif_albums(albums))
        for (p, cw, ch, d, pl), outs in zip(albums, got):
            for g, a in zip(outs, gpu.gif_album(p, cw, ch, d, pl)):
                assert np.array_equal(g, a), (cw, ch)
        rounds = round_bounds(shim, geoms)
        assert len(rounds) - 1 >= 3
        replay = [(p, cw, ch, d, [None] * len(p)) for p, cw, ch, d, _ in albums]
        before = gpu.launch_count()
        gpu.gif_albums(replay)
        assert gpu.launch_count() - before == len(rounds) - 1
    finally:
        for p in plans.values():
            p.close()


@pytest.mark.gpu
@pytest.mark.parametrize("defect", ["plan_geometry", "null_pages", "no_pages", "short_dst_step"])
def test_bad_album_writes_nothing(gpu, defect):
    rng = np.random.default_rng(53)
    cw, ch, n = 64, 48, 4
    plan = _plan(gpu, cw, ch, dict(resize="32,24", simple=True))
    wrong = _plan(gpu, cw + 1, ch, dict(resize="32,24", simple=True))
    try:
        albums = []
        for i in range(5):
            outs = [np.full((24, 32, 4), 0xA5, np.uint8) for _ in range(n)]
            albums.append((_pages(rng, cw, ch, n, padded=False), cw, ch, True, plan, outs))
        job = api.GifAlbumsJob(gpu, albums)
        mid = job.arr[2]
        if defect == "plan_geometry":
            job.jobs[2].P[1] = wrong.h
        elif defect == "null_pages":
            mid.pages = None
        elif defect == "no_pages":
            mid.n_pages = 0
        else:
            job.jobs[2].DS[3] = 32 * 4 - 1
        with pytest.raises(api.ImpError) as e:
            job.run(gpu)
        assert e.value.code == api.IMP_ERROR_INVALID_ARGS
        for a in albums:
            for o in a[5]:
                assert (o == 0xA5).all(), defect
    finally:
        plan.close()
        wrong.close()


@pytest.mark.gpu
def test_no_albums(gpu):
    assert gpu.gif_albums([]) == []


DBG_SCRIPT = r"""
import sys, ctypes as C, numpy as np
sys.path.insert(0, "."); sys.path.insert(0, "tests")
import ngx_http_imgproc_b200 as M
import test_gif_albums as T
L = M.library(); L.init(0)
L.lib.imp_gpu_debug_flags.restype = C.c_uint
albums, plans, rqs = T._mixed(L, np.random.default_rng(41))
got = T._copy(L.gif_albums(albums))
for (pages, cw, ch, d, per), outs in zip(albums, got):
    for g, a in zip(outs, L.gif_album(pages, cw, ch, d, per)):
        assert (g is None and a is None) or np.array_equal(g, a)
flags = L.lib.imp_gpu_debug_flags()
print("DBG", hex(flags))
assert flags == 0, hex(flags)
"""


@pytest.mark.gpu
def test_mixed_albums_debug_build():
    """The mixed batch over libimp_gpu_dbg.so (bounds assertions on every index-plane and canvas address the expansion
    forms), in a child process: no assertion fires and the results still equal one call per album."""
    dbg = os.path.join(ROOT, "ngx_http_imgproc_b200", "libimp_gpu_dbg.so")
    assert os.path.exists(dbg), "the debug library is built by __graft_entry__.build()"
    r = subprocess.run([sys.executable, "-c", DBG_SCRIPT], cwd=ROOT, env=dict(os.environ, IMP_GPU_LIB=dbg), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "DBG 0x0" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]
