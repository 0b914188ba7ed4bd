"""CPU tests of how the chunked host path moves a batch over the link (imp_transfer.cpp): where a batch is cut into chunks
(imp_chunk_bounds) and, per job of a chunk, the route its source takes to the device and its result back to the host, with
the offsets of both in the lane's buffers (imp_chunk_layout). The expected values restate the rules independently:

* chunks: n_streams clamped to 1..8; at most max(1, min(256, ceil(n / n_streams))) jobs and, beyond a chunk's first job,
  at most min(128 MB, max(4 MB, total / (2 n_streams))) bytes, where a job moves align16(win_w*src_c)*win_h bytes of crop
  window and out_w*out_c*out_h bytes of result;
* sources: Resident when already on the device; Staged when pageable (4 row slices for a lone job of 16 MB or more, else
  1); pinned: Linear when step == in_pitch and win_x == 0 and (step <= 8192 or the window row is its pitch), else
  LinearRepitch when step <= 8192, else Rows2D;
* results: pageable -> Staged; pinned frames -> Linear when dst_step == out_pitch, else Rows2D; pinned answers -> Direct;
* every offset 256-byte aligned, except staged brightness floats, packed 4 bytes apart."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RESIDENT, STAGED, LINEAR, LINEAR_REPITCH, ROWS_2D, DIRECT = range(6)        # ImpRoute (imp_internal.h)
FRAME, BRIGHTNESS, ASCII = range(3)                                         # ImpResult
MB = 1 << 20
FIELDS = ("src", "dst", "in_pitch", "out_pitch", "in_off", "out_off", "lin_bytes", "stage_off", "hin_off", "hout_off", "res_bytes", "slices")


def a16(v):
    return (v + 15) & ~15


def a256(v):
    return (v + 255) & ~255


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("transfer") / "libtransfer_shim.so")
    cuda_inc = os.environ.get("CUDA_HOME", "/usr/local/cuda") + "/include"
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-w", "-I" + cuda_inc, "-o", so,
                    os.path.join(ROOT, "tests", "hostsim", "transfer_shim.cpp"),
                    os.path.join(ROOT, "ngx_http_imgproc_b200", "csrc", "imp_transfer.cpp")], check=True)
    lib = C.CDLL(so)
    lib.shim_plan.restype = C.c_void_p
    lib.shim_plan.argtypes = [C.c_int] * 10
    lib.shim_plan_free.argtypes = [C.c_void_p]
    lib.shim_bounds.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_void_p]
    lib.shim_layout.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    return lib


class Job:
    """A job's geometry: source (w, h, c), crop window (x, y, w, h), result (w, h, c), and its steps."""

    def __init__(self, src, win, out, src_step=None, dst_step=None):
        self.src, self.win, self.out = src, win, out
        self.src_step = src[0] * src[2] if src_step is None else src_step
        self.dst_step = out[0] * out[2] if dst_step is None else dst_step

    in_row = property(lambda s: s.win[2] * s.src[2])
    out_row = property(lambda s: s.out[0] * s.out[2])
    bytes = property(lambda s: a16(s.in_row) * s.win[3] + s.out_row * s.out[1])


def _plans(shim, jobs):
    ps = [shim.shim_plan(*j.src, *j.win, *j.out) for j in jobs]
    return ps, (C.c_void_p * max(len(ps), 1))(*ps)


def bounds(shim, jobs, n_streams):
    ps, P = _plans(shim, jobs)
    out = (C.c_int * (len(jobs) + 2))()
    k = shim.shim_bounds(len(jobs), P, n_streams, out)
    for p in ps:
        shim.shim_plan_free(p)
    return list(out[:k])


def layout(shim, jobs, kind, src_pinned, dst_pinned, resident=False):
    m = len(jobs)
    ps, P = _plans(shim, jobs)
    ss = (C.c_int * m)(*[j.src_step for j in jobs])
    ds = (C.c_int * m)(*[j.dst_step for j in jobs])
    sp = (C.c_ubyte * m)(*[1 if x else 0 for x in src_pinned])
    dp = (C.c_ubyte * m)(*[1 if x else 0 for x in dst_pinned])
    per, tot = (C.c_longlong * (12 * m))(), (C.c_longlong * 5)()
    shim.shim_layout(m, P, ss, ds, kind, 1 if resident else 0, sp, dp, per, tot)
    for p in ps:
        shim.shim_plan_free(p)
    return [dict(zip(FIELDS, per[12 * k:12 * k + 12])) for k in range(m)], list(tot)


def expected_bounds(jobs, n_streams):
    n_streams = max(1, min(n_streams, 8))
    n = len(jobs)
    chunk_bytes = min(128 * MB, max(4 * MB, sum(j.bytes for j in jobs) // (2 * n_streams)))
    max_jobs = max(1, min(256, -(-n // n_streams)))
    b, i = [0], 0
    while i < n:
        e, acc = i, 0
        while e < n and e - i < max_jobs and (e == i or acc + jobs[e].bytes <= chunk_bytes):
            acc += jobs[e].bytes
            e += 1
        b.append(e)
        i = e
    return b


def expected_src(j, pinned, resident=False):
    if resident:
        return RESIDENT
    if not pinned:
        return STAGED
    pitch = a16(j.in_row)
    if j.src_step == pitch and j.win[0] == 0 and (j.src_step <= 8192 or j.in_row == pitch):
        return LINEAR
    return LINEAR_REPITCH if j.src_step <= 8192 else ROWS_2D


def expected_dst(j, kind, pinned):
    if not pinned:
        return STAGED
    if kind != FRAME:
        return DIRECT
    return LINEAR if j.dst_step == a16(j.out_row) else ROWS_2D


def source_matrix():
    """Pinned source cases over short (<= 8192 B) and long rows, windows at x == 0 and not, window rows equal to their
    16-byte pitch and not, frame steps dense, 16-byte padded and wider."""
    cases = []
    for w in (200, 1000, 2900, 3000):
        for c in (3, 4):
            row = w * c
            for (wx, ww) in ((0, w), (0, w - 4), (8, w - 16), (3, w - 7)):
                for step in sorted({row, a16(row), row + 64}):
                    cases.append(Job((w, 40, c), (wx, 5, ww, 30), (ww // 2, 15, c), src_step=step))
    return cases


def test_source_routes_over_the_matrix(shim):
    jobs = source_matrix()
    seen = set()
    for pinned in (True, False):
        for j in jobs:
            got = layout(shim, [j], FRAME, [pinned], [True])[0][0]
            want = expected_src(j, pinned)
            assert got["src"] == want, (j.src, j.win, j.src_step, pinned, got["src"], want)
            seen.add(want)
    j = jobs[0]
    assert layout(shim, [j, j], FRAME, [False, True], [True, True], resident=True)[0][0]["src"] == RESIDENT
    assert seen == {STAGED, LINEAR, LINEAR_REPITCH, ROWS_2D}
    # the boundary rows: a window that is the frame's contiguous rows is one linear copy at any length; a padded one above
    # 8192 bytes is a 2-D copy
    long_dense = Job((3000, 20, 4), (0, 0, 3000, 20), (100, 10, 4))
    assert long_dense.src_step == 12000 and layout(shim, [long_dense], FRAME, [True], [True])[0][0]["src"] == LINEAR
    long_padded = Job((2731, 20, 3), (0, 0, 2731, 20), (100, 10, 3), src_step=a16(8193))
    assert layout(shim, [long_padded], FRAME, [True], [True])[0][0]["src"] == ROWS_2D
    short_padded = Job((2730, 20, 3), (0, 0, 2730, 20), (100, 10, 3), src_step=8192)
    assert layout(shim, [short_padded], FRAME, [True], [True])[0][0]["src"] == LINEAR


@pytest.mark.parametrize("kind", [FRAME, BRIGHTNESS, ASCII])
def test_destination_routes(shim, kind):
    for (w, c) in ((100, 3), (64, 4), (33, 1)):
        row = w * c
        for step in sorted({row, a16(row), row + 100}):
            j = Job((400, 300, 3), (0, 0, 400, 300), (w, 50, c), dst_step=step)
            for pinned in (True, False):
                got = layout(shim, [j], kind, [True], [pinned])[0][0]
                assert got["dst"] == expected_dst(j, kind, pinned), (kind, w, c, step, pinned)


def mixed_chunk():
    return [Job((640, 480, 3), (0, 0, 640, 480), (320, 240, 3)),                                  # dense pinned: Linear
            Job((640, 480, 3), (17, 9, 501, 400), (250, 200, 3), dst_step=256 * 3 + 16),          # short rows: LinearRepitch
            Job((4000, 300, 3), (5, 2, 3990, 290), (1000, 70, 3)),                                # long rows: Rows2D
            Job((333, 211, 4), (1, 1, 331, 209), (331, 209, 4), dst_step=331 * 4 + 4),            # pageable in and out
            Job((1920, 1080, 3), (0, 0, 1920, 1080), (640, 360, 3)),                              # pageable source
            Job((97, 13, 1), (3, 0, 91, 13), (45, 6, 1))]                                         # pageable result


@pytest.mark.parametrize("kind", [FRAME, BRIGHTNESS, ASCII])
def test_offsets_are_aligned_disjoint_and_add_up(shim, kind):
    jobs = mixed_chunk()
    src_pinned = [True, True, True, False, False, True]
    dst_pinned = [True, True, True, False, True, False] if kind != BRIGHTNESS else [False] * 6
    lay, tot = layout(shim, jobs, kind, src_pinned, dst_pinned)
    assert [l["src"] for l in lay] == [LINEAR, LINEAR_REPITCH, ROWS_2D, STAGED, STAGED, LINEAR_REPITCH]
    regions = {"in": [], "out": [], "stage": [], "hin": [], "hout": []}
    for j, l, sp, dp in zip(jobs, lay, src_pinned, dst_pinned):
        in_pitch, out_pitch = a16(j.in_row), a16(j.out_row)
        assert (l["in_pitch"], l["out_pitch"]) == (in_pitch, out_pitch)
        assert l["src"] == expected_src(j, sp) and l["dst"] == expected_dst(j, kind, dp)
        res = j.out_row * j.out[1] if kind == FRAME else 4 if kind == BRIGHTNESS else (j.out[0] + 1) * j.out[1] - 1
        assert l["res_bytes"] == res
        regions["in"].append((l["in_off"], in_pitch * j.win[3]))
        regions["out"].append((l["out_off"], out_pitch * j.out[1]))
        if l["src"] in (LINEAR, LINEAR_REPITCH):
            assert l["lin_bytes"] == (j.win[3] - 1) * j.src_step + j.win[0] * j.src[2] + j.in_row
        if l["src"] == LINEAR_REPITCH:
            regions["stage"].append((l["stage_off"], l["lin_bytes"]))
        if l["src"] == STAGED:
            regions["hin"].append((l["hin_off"], in_pitch * j.win[3]))
            assert l["slices"] == 1                                       # several jobs: never sliced
        if l["dst"] == STAGED:
            regions["hout"].append((l["hout_off"], res))
    for name, regs in regions.items():
        packed = name == "hout" and kind == BRIGHTNESS
        end = 0
        for off, size in regs:                                            # in job order, each after the previous one
            assert off >= end, (name, regs)
            assert off % (4 if packed else 256) == 0, (name, off)
            end = off + (size if packed else a256(size))
        if packed:
            assert [off for off, _ in regs] == [4 * k for k in range(len(regs))]
    assert tot == [sum(a256(s) for _, s in regions[r]) if not (r == "hout" and kind == BRIGHTNESS) else 4 * len(regions[r])
                   for r in ("in", "out", "stage", "hin", "hout")]
    # resident sources need no landing zone
    lay_r, tot_r = layout(shim, jobs, kind, [True] * 6, dst_pinned, resident=True)
    assert tot_r[0] == 0 and tot_r[2] == 0 and tot_r[3] == 0 and tot_r[1] == tot[1]
    assert all(l["src"] == RESIDENT for l in lay_r)


def test_brightness_answers_of_a_chunk_share_one_route(shim):
    """Brightness floats are one array: the first job's pinnedness decides for the chunk (one copy back)."""
    jobs = mixed_chunk()
    for first in (True, False):
        lay, _ = layout(shim, jobs, BRIGHTNESS, [True] * 6, [first] + [not first] * 5)
        assert {l["dst"] for l in lay} == {DIRECT if first else STAGED}


def test_a_lone_pageable_window_is_sliced_from_16_mb(shim):
    def slices(jobs):
        return [l["slices"] for l in layout(shim, jobs, FRAME, [False] * len(jobs), [True] * len(jobs))[0]]
    below = Job((2048, 2048, 4), (0, 0, 2048, 2047), (64, 64, 4))       # 2048*4*2047 bytes: just under 16 MB
    at = Job((2048, 2048, 4), (0, 0, 2048, 2048), (64, 64, 4))          # exactly 16 MB
    cfg2 = Job((3840, 2160, 4), (120, 67, 3600, 2025), (800, 450, 4))   # 29 MB
    assert below.in_row * below.win[3] < 16 * MB <= at.in_row * at.win[3]
    assert slices([below]) == [1] and slices([at]) == [4] and slices([cfg2]) == [4]
    assert slices([cfg2, cfg2]) == [1, 1]
    tall_row = Job((3 << 20, 3, 3), (0, 0, 3 << 20, 3), (8, 1, 3))        # 3 rows of 9 MB: one slice per row
    assert slices([tall_row]) == [3]


def _bench_jobs(name):
    """The e2e shapes of bench.py (cfg5: its 4096-job sample, every 16th job of the 65536), geometry from the planner."""
    import bench
    import ngx_http_imgproc_b200 as M
    from ngx_http_imgproc_b200 import api
    L = M.library()
    wl = bench.workload(name, 1)
    cfg = api.Config(**wl["cfg"])
    geo = []
    for (h, w, c), rq, _ in wl["jobs"]:
        p = L.plan(w, h, c, cfg, **rq)
        geo.append(Job((w, h, c), tuple(p.window), (p.out_w, p.out_h, p.out_c)))
        p.close()
    order = bench.job_order(wl)
    if len(order) > 4096:
        order = order[::max(1, len(order) // 4096)][:4096]
    return [geo[i] for i in order]


def test_chunk_bounds_of_the_bench_shapes(shim):
    cfg1, cfg2, cfg4, cfg5 = (_bench_jobs(n) for n in ("cfg1", "cfg2", "cfg4", "cfg5"))
    # cfg1: 6.9 MB a job, 128 MB chunks -> 19 jobs; cfg2: 30.6 MB a job -> 4 jobs; cfg4: 72 MB a job, 8 jobs over 4 lanes
    # -> 72 MB chunks (total / 8) of one job each
    assert cfg1[0].bytes == 6912000 and bounds(shim, cfg1, 4) == list(range(0, 256, 19)) + [256]
    assert cfg2[0].bytes == 30600000 and bounds(shim, cfg2, 4) == list(range(0, 257, 4))
    assert cfg4[0].bytes == 72000000 and bounds(shim, cfg4, 4) == list(range(9))
    assert len(cfg5) == 4096
    got = bounds(shim, cfg5, 4)
    assert got == expected_bounds(cfg5, 4)
    assert got[0] == 0 and got[-1] == 4096 and all(b - a <= 256 for a, b in zip(got, got[1:]))


def test_chunk_bounds_of_small_batches(shim):
    tiny = Job((23, 17, 3), (0, 0, 23, 17), (9, 7, 3))
    mb = Job((512, 512, 4), (0, 0, 512, 480), (128, 128, 4))           # about 1 MB a job
    assert bounds(shim, [], 4) == [0]
    assert bounds(shim, [tiny], 4) == [0, 1]
    assert bounds(shim, [tiny] * 3, 4) == [0, 1, 2, 3]                  # spread over the lanes
    assert bounds(shim, [tiny] * 10, 4) == [0, 3, 6, 9, 10]
    assert bounds(shim, [tiny] * 40, 4) == list(range(0, 41, 10))
    assert bounds(shim, [tiny] * 600, 1) == [0, 256, 512, 600]          # at most 256 jobs a chunk
    assert bounds(shim, [tiny] * 100, 0) == [0, 100]                    # n_streams clamped to 1..8
    assert bounds(shim, [tiny] * 100, 50) == list(range(0, 100, 13)) + [100]
    # 40 MB over 4 lanes: 5 MB chunks (total / 8), so 5 jobs each
    assert 40 * MB // 8 // mb.bytes == 5 and bounds(shim, [mb] * 40, 4) == list(range(0, 41, 5))
    # a job larger than a chunk still makes a chunk of its own
    huge = Job((16000, 12000, 3), (0, 0, 16000, 12000), (16000, 12000, 3))
    assert bounds(shim, [tiny, huge, tiny], 1) == [0, 1, 2, 3]
    rng = np.random.default_rng(7)
    for it in range(20):
        jobs = [Job((int(w), int(h), 3), (0, 0, int(w), int(h)), (int(w) // 2, int(h) // 2, 3))
                for w, h in rng.integers(16, 3000, (int(rng.integers(1, 300)), 2))]
        ns = int(rng.integers(1, 9))
        assert bounds(shim, jobs, ns) == expected_bounds(jobs, ns), it
