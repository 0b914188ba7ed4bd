"""Submit / poll / wait for every host call: imp_gpu_batch_submit_host (frames), imp_gpu_batch_brightness_submit_host
(format=json), imp_gpu_batch_ascii_submit_host (format=text) and imp_gpu_gif_albums_submit_host (GIF requests).

CPU: a C99 host calls the three answer and album submits with no device initialised: IMP_ERROR_GPU, no ticket, nothing
written; a NULL ticket argument is an argument error.

GPU: each submit gives exactly what its synchronous twin gives, and the oracle, at n_streams 1 and 4; tickets of every kind
in flight at once, from one thread and from four; a submit returns before its work is done; every defect the synchronous
calls refuse is refused at the submit with nothing written; the caller's argument arrays and plans may go right after the
submit; the work runs on the device that was current at the submit; the album submit on the debug build."""
import ctypes as C
import os
import subprocess
import sys
import threading
import time

import numpy as np
import pytest

import ngx_http_imgproc_b200 as M
from ngx_http_imgproc_b200 import api
import golden_util as G
import test_gif_albums as GA
import test_info_outputs as IO
from conftest import ROOT, rnd_image, smooth_image
from test_planner_host import _oracle


def test_a_c_host_gets_no_ticket_without_a_device(tmp_path):
    src = tmp_path / "submit.c"
    src.write_text(r'''
#include <stdio.h>
#include <string.h>
#include "imp_gpu.h"
static unsigned char px[48 * 64 * 4], text[2 * 1024], idx[48 * 64], pal[1024], out[24 * 32 * 4];
int main(void) {
    imp_gpu_request rq; imp_gpu_config cfg; imp_gpu_plan *plan = NULL, *gplan = NULL; int step = -1, i;
    imp_gpu_ticket* const junk = (imp_gpu_ticket*)(void*)px;
    imp_gpu_ticket* t;
    float bright[2] = {-7.0f, -7.0f};
    memset(&rq, 0, sizeof rq); memset(&cfg, 0, sizeof cfg);
    cfg.max_filters = 5; rq.resize = "32,24";
    if (imp_gpu_plan_create(&rq, &cfg, 64, 48, 3, &plan, &step) != IMP_OK) return 1;
    if (imp_gpu_plan_create(&rq, &cfg, 64, 48, 4, &gplan, &step) != IMP_OK) return 2;
    memset(text, 0x5a, sizeof text); memset(out, 0x5a, sizeof out);
    {
        imp_gpu_plan* plans[2]; const unsigned char* srcs[2]; int steps[2] = {64 * 3, 64 * 3};
        const char* args[2] = {"wide", NULL}; unsigned char* texts[2]; long caps[2] = {1024, 1024};
        imp_gpu_gif_frame page; imp_gpu_gif_album album;
        imp_gpu_plan* gplans[1]; unsigned char* dsts[1]; int dst_steps[1] = {32 * 4};
        plans[0] = plans[1] = plan; srcs[0] = srcs[1] = px; texts[0] = text; texts[1] = text + 1024;
        gplans[0] = gplan; dsts[0] = out;
        memset(&page, 0, sizeof page);
        page.indices = idx; page.pitch = 64; page.width = 64; page.height = 48; page.transparency_key = -1; page.palette = pal;
        album.pages = &page; album.n_pages = 1; album.canvas_w = 64; album.canvas_h = 48; album.destructive = 1;
        album.plans = gplans; album.dsts = dsts; album.dst_steps = dst_steps;
        t = junk; if (imp_gpu_batch_brightness_submit_host(2, plans, srcs, steps, bright, 4, &t) != IMP_ERROR_GPU || t) return 10;
        t = junk; if (imp_gpu_batch_ascii_submit_host(2, plans, srcs, steps, args, texts, caps, 4, &t) != IMP_ERROR_GPU || t) return 11;
        t = junk; if (imp_gpu_gif_albums_submit_host(&album, 1, 4, &t) != IMP_ERROR_GPU || t) return 12;
        if (strlen(imp_gpu_last_error()) == 0) return 13;
        if (imp_gpu_batch_brightness_submit_host(2, plans, srcs, steps, bright, 4, NULL) != IMP_ERROR_INVALID_ARGS) return 14;
        if (imp_gpu_batch_ascii_submit_host(2, plans, srcs, steps, args, texts, caps, 4, NULL) != IMP_ERROR_INVALID_ARGS) return 15;
        if (imp_gpu_gif_albums_submit_host(&album, 1, 4, NULL) != IMP_ERROR_INVALID_ARGS) return 16;
    }
    if (bright[0] != -7.0f || bright[1] != -7.0f) return 20;
    for (i = 0; i < (int)sizeof text; i++) if (text[i] != 0x5a) return 21;
    for (i = 0; i < (int)sizeof out; i++) if (out[i] != 0x5a) return 22;
    imp_gpu_plan_destroy(plan); imp_gpu_plan_destroy(gplan);
    printf("SUBMIT HOST OK\n");
    return 0;
}
''')
    exe = tmp_path / "submit"
    pkg = os.path.join(ROOT, "ngx_http_imgproc_b200")
    M.build()
    r = subprocess.run(["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src),
                        "-L", pkg, "-limp_gpu", "-Wl,-rpath," + pkg], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0 and "SUBMIT HOST OK" in r.stdout, (r.returncode, r.stdout, r.stderr)


# ---- on the GPU -------------------------------------------------------------------------------------------------------
def _images(seed):
    return [smooth_image(seed + k, *shape) if k % 2 else rnd_image(seed + k, *shape) for k, (shape, _, _) in enumerate(IO.CASES)]


def _plans(gpu):
    imgs = _images(0)
    return [gpu.plan(i.shape[1], i.shape[0], i.shape[2], api.Config(**kw), **rq) for i, (_, kw, rq) in zip(imgs, IO.CASES)]


ARGS = ["wide" if k % 2 else None for k in range(len(IO.CASES))]


def _wait(gpu, ticket):
    api.HostJobs.wait(gpu, ticket)


@pytest.mark.gpu
@pytest.mark.parametrize("n_streams", [1, 4])
def test_album_submit_equals_the_call_and_the_oracle(gpu, orc, n_streams):
    """The mixed album set of test_gif_albums: the submit's bytes equal the synchronous call's, which equal the oracle's."""
    o = orc.orc()
    albums, plans, rqs = GA._mixed(gpu, np.random.default_rng(41))
    try:
        want = GA._copy(gpu.gif_albums(albums, n_streams=n_streams))
        job = api.GifAlbumsJob(gpu, albums)
        t = job.submit(gpu, n_streams)
        _wait(gpu, t)
        GA._assert_albums_equal(job.outs, want, "submit")
        for (pages, cw, ch, d, per), rq, outs in zip(albums, rqs, want):
            canvases = o.gif_expand(pages, cw, ch, d)
            for f, g in enumerate(outs):
                if per[f] is not None:
                    code, _, ref = _oracle(orc, canvases[f], rq, {})
                    assert code == 0 and g.shape == ref.shape and np.array_equal(g, ref), (cw, ch, rq, f)
    finally:
        for p in plans:
            p.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n_streams", [1, 4])
def test_answer_submits_equal_the_calls_and_the_oracle(gpu, orc, n_streams):
    """The mixed batch of test_info_outputs: the same brightness bits and the same texts as the synchronous calls, and those
    against the oracle as test_info_outputs holds them."""
    imgs, plans = _images(0), _plans(gpu)
    try:
        b_want = gpu.batch_brightness(plans, imgs, n_streams=n_streams)
        t_want = gpu.batch_ascii(plans, imgs, ARGS, n_streams=n_streams)
        tb, b = gpu.batch_brightness_submit(plans, imgs, n_streams)
        ta, texts = gpu.batch_ascii_submit(plans, imgs, ARGS, n_streams)
        _wait(gpu, ta)
        _wait(gpu, tb)
        assert b.tobytes() == b_want.tobytes()
        assert [x.tobytes() for x in texts] == t_want
        frames = IO._frames(gpu, plans, imgs)
        o = orc.orc()
        for k, ((shape, kw, rq), img, fr) in enumerate(zip(IO.CASES, imgs, frames)):
            code, _, ref = _oracle(orc, img, rq, kw)
            assert code == 0
            if IO._vignette(rq):
                G.assert_vignette_exact(fr, ref, shape, kw, rq, (k, rq))
            assert IO._within_one_ulp(b[k], IO._numpy_brightness(fr)), (k, rq)
            assert abs(float(b[k]) - o.perceived_brightness(ref)) < 1e-4, (k, rq)
            assert texts[k].tobytes() == o.ascii(fr if IO._vignette(rq) else ref, ARGS[k] == "wide"), (k, rq)
    finally:
        IO._close(plans)


class Mix:
    """One ticket of every kind over shared plans: a frame batch, a brightness batch, an ASCII batch and an album batch, with
    the synchronous results each must equal."""

    def __init__(self, gpu, plans, gplan, seed):
        self.plans, self.imgs = plans, _images(100 * seed)
        rng = np.random.default_rng(seed)
        self.albums = [(GA._pages(rng, 160, 120, 6, padded=bool(i % 2)), 160, 120, i % 2 == 0, gplan) for i in range(5)]
        self.frames = IO._frames(gpu, plans, self.imgs)
        self.bright = gpu.batch_brightness(plans, self.imgs)
        self.texts = gpu.batch_ascii(plans, self.imgs, ARGS)
        self.album_outs = GA._copy(gpu.gif_albums(self.albums))

    def submit(self, gpu, n_streams):
        outs = [np.zeros_like(f) for f in self.frames]
        tf = api.HostJobs(self.plans, self.imgs, outs).submit(gpu, n_streams)
        tb, b = gpu.batch_brightness_submit(self.plans, self.imgs, n_streams)
        ta, texts = gpu.batch_ascii_submit(self.plans, self.imgs, ARGS, n_streams)
        job = api.GifAlbumsJob(gpu, self.albums)
        tg = job.submit(gpu, n_streams)
        return [tf, tb, ta, tg], (outs, b, texts, job)

    def check(self, got, what):
        outs, b, texts, job = got
        assert all(np.array_equal(x, y) for x, y in zip(outs, self.frames)), what
        assert b.tobytes() == self.bright.tobytes(), what
        assert [x.tobytes() for x in texts] == self.texts, what
        GA._assert_albums_equal(job.outs, self.album_outs, what)


@pytest.mark.gpu
def test_tickets_of_every_kind_in_flight_from_one_thread(gpu):
    plans, gplan = _plans(gpu), GA._plan(gpu, 160, 120, dict(resize="80,60", **GA.NN_SEPIA))
    try:
        mix = Mix(gpu, plans, gplan, 1)
        tickets, got = mix.submit(gpu, 4)
        for t in tickets[::-1]:
            _wait(gpu, t)
        mix.check(got, "one thread")
    finally:
        IO._close(plans + [gplan])


@pytest.mark.gpu
def test_tickets_of_every_kind_in_flight_from_four_threads(gpu):
    plans, gplan = _plans(gpu), GA._plan(gpu, 160, 120, dict(resize="80,60", **GA.NN_SEPIA))
    errors = []
    try:
        mixes = [Mix(gpu, plans, gplan, 2 + t) for t in range(4)]

        def worker(t):
            try:
                for it in range(3):
                    tickets, got = mixes[t].submit(gpu, 1 + (t + it) % 4)
                    for tk in tickets[::-1]:
                        _wait(gpu, tk)
                    mixes[t].check(got, (t, it))
            except Exception as e:                                       # noqa: BLE001 — reported by the main thread
                errors.append(repr(e))

        threads = [threading.Thread(target=worker, args=(t,)) for t in range(4)]
        for th in threads:
            th.start()
        for th in threads:
            th.join(timeout=600)
        assert not any(th.is_alive() for th in threads)
        assert not errors, errors[:3]
    finally:
        IO._close(plans + [gplan])


@pytest.mark.gpu
def test_an_album_submit_returns_before_its_work_is_done(gpu):
    """Albums of 640x480 pages (one page set shared by every album) whose synchronous call takes 100 ms or more: the submit
    returns while the work runs, before any destination is written, and the destinations are exact after the wait."""
    cw, ch, n = 640, 480, 40
    rng = np.random.default_rng(61)
    pages = [dict(indices=rng.integers(0, 256, (ch, cw), dtype=np.uint8), left=0, top=0, dispose=int(rng.integers(0, 4)),
                  key=int(rng.integers(-1, 256)), palette=rng.integers(0, 256, (256, 4), dtype=np.uint8)) for _ in range(n)]
    plan = GA._plan(gpu, cw, ch, dict(resize="80,60", filters=["modulate=0,0,100", "colorize=704214,0.6"]))
    try:
        ref = np.stack(gpu.gif_album(pages, cw, ch, True, plan))

        def make(k):
            big = np.full((k, n, 60, 80, 4), 0xA5, np.uint8)
            return big, api.GifAlbumsJob(gpu, [(pages, cw, ch, True, plan, list(big[a])) for a in range(k)])

        k = 32
        for _ in range(3):                                            # grow the set until the call takes 100 ms or more
            big, job = make(k)
            job.run(gpu, 1)
            t0 = time.perf_counter()
            job.run(gpu, 1)
            sync = time.perf_counter() - t0
            if sync >= 0.1:
                break
            k = min(int(k * 0.15 / sync) + 1, 600)
        assert sync >= 0.1, (k, sync)
        big[...] = 0xA5
        t0 = time.perf_counter()
        t = job.submit(gpu, 1)
        took = time.perf_counter() - t0
        running = not api.HostJobs.poll(gpu, t)
        first_untouched = bool((big[0] == 0xA5).all())
        _wait(gpu, t)
        assert running and first_untouched, (running, first_untouched, took, sync)
        assert took < sync / 4, (took, sync)
        assert (big == ref[None]).all()
    finally:
        plan.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["null_plan", "short_src_step", "short_dst_step", "packed", "small_caps", "null_arrays"])
def test_a_bad_job_is_refused_at_the_submit(gpu, case):
    """The defects test_gpu_host_path and test_info_outputs give the synchronous calls (a NULL plan in the last chunk, a
    short source or destination step, a packed answer, a text capacity one byte short, NULL argument arrays): each submit
    returns its twin's code, no ticket, and every output as it was."""
    L = gpu.lib
    n, bad = 40, 39
    imgs = [rnd_image(200 + i, 48, 64, 3) for i in range(n)]
    plan = gpu.plan(64, 48, 3, api.Config(max_w=0, max_h=0), resize="32,24")
    packed = gpu.plan(64, 48, 3, resize="40,30", pack=24)
    try:
        row = plan.out_w * plan.out_c
        k = L.imp_gpu_ascii_length(plan.out_w, plan.out_h)
        P = (C.c_void_p * n)(*[None if (case == "null_plan" and i == bad) else (packed if (case == "packed" and i == bad) else plan).h.value
                              for i in range(n)])
        S = (C.c_void_p * n)(*[im.ctypes.data for im in imgs])
        SS = (C.c_int * n)(*[im.strides[0] - (1 if (case == "short_src_step" and i == bad) else 0) for i, im in enumerate(imgs)])
        dsts = [np.full((plan.out_h, row), 0x5a, np.uint8) for _ in range(n)]
        D = (C.c_void_p * n)(*[d.ctypes.data for d in dsts])
        DS = (C.c_int * n)(*[row - (1 if (case == "short_dst_step" and i == bad) else 0) for i in range(n)])
        b = np.full(n, -7.0, np.float32)
        texts = [np.full(k, 0x5a, np.uint8) for _ in range(n)]
        T = (C.c_void_p * n)(*[x.ctypes.data for x in texts])
        A = (C.c_char_p * n)(*[b"wide"] * n)
        caps = (C.c_long * n)(*[k - (1 if (case == "small_caps" and i == bad) else 0) for i in range(n)])
        nul = case == "null_arrays"
        calls = [("frames", lambda: L.imp_gpu_batch_run_host(n, None if nul else P, S, SS, D, DS, 4),
                  lambda t: L.imp_gpu_batch_submit_host(n, None if nul else P, S, SS, D, DS, 4, t),
                  lambda: all((d == 0x5a).all() for d in dsts)),
                 ("brightness", lambda: L.imp_gpu_batch_brightness_host(n, P, S, None if nul else SS, b.ctypes.data, 4),
                  lambda t: L.imp_gpu_batch_brightness_submit_host(n, P, S, None if nul else SS, b.ctypes.data, 4, t),
                  lambda: (b == -7.0).all()),
                 ("ascii", lambda: L.imp_gpu_batch_ascii_host(n, P, S, SS, A, T, None if nul else caps, 4),
                  lambda t: L.imp_gpu_batch_ascii_submit_host(n, P, S, SS, A, T, None if nul else caps, 4, t),
                  lambda: all((x == 0x5a).all() for x in texts))]
        refused = 0
        for what, sync, submit, untouched in calls:
            want = sync()
            if want == M.IMP_OK:                                      # a defect this call does not see (an answer has no step)
                continue
            assert want == M.IMP_ERROR_INVALID_ARGS and untouched(), (case, what, want)
            t = C.c_void_p(12345)
            assert submit(C.byref(t)) == want and not t.value and untouched(), (case, what)
            refused += 1
        assert refused >= 1
    finally:
        plan.close()
        packed.close()


@pytest.mark.gpu
@pytest.mark.parametrize("defect", ["plan_geometry", "null_pages", "no_pages", "short_dst_step"])
def test_a_bad_album_is_refused_at_the_submit(gpu, defect):
    """Every defect of test_gif_albums.test_bad_album_writes_nothing, in the middle album of five."""
    rng = np.random.default_rng(53)
    cw, ch, n = 64, 48, 4
    plan = GA._plan(gpu, cw, ch, dict(resize="32,24", simple=True))
    wrong = GA._plan(gpu, cw + 1, ch, dict(resize="32,24", simple=True))
    try:
        albums = [(GA._pages(rng, cw, ch, n, padded=False), cw, ch, True, plan, [np.full((24, 32, 4), 0xA5, np.uint8) for _ in range(n)])
                  for _ in range(5)]
        job = api.GifAlbumsJob(gpu, albums)
        if defect == "plan_geometry":
            job.jobs[2].P[1] = wrong.h
        elif defect == "null_pages":
            job.arr[2].pages = None
        elif defect == "no_pages":
            job.arr[2].n_pages = 0
        else:
            job.jobs[2].DS[3] = 32 * 4 - 1
        want = gpu.lib.imp_gpu_gif_albums_run_host(job.arr, job.n, 4)
        assert want == M.IMP_ERROR_INVALID_ARGS
        t = C.c_void_p(12345)
        assert gpu.lib.imp_gpu_gif_albums_submit_host(job.arr, job.n, 4, C.byref(t)) == want and not t.value
        assert all((o == 0xA5).all() for a in albums for o in a[5]), defect
    finally:
        plan.close()
        wrong.close()


@pytest.mark.gpu
def test_no_jobs_give_a_ticket_that_waits_ok(gpu):
    L = gpu.lib
    for call in (lambda t: L.imp_gpu_batch_brightness_submit_host(0, None, None, None, None, 4, t),
                 lambda t: L.imp_gpu_batch_ascii_submit_host(0, None, None, None, None, None, None, 4, t),
                 lambda t: L.imp_gpu_gif_albums_submit_host(None, 0, 4, t)):
        t = C.c_void_p()
        assert call(C.byref(t)) == M.IMP_OK and t.value
        assert L.imp_gpu_batch_wait(t) == M.IMP_OK


@pytest.mark.gpu
def test_the_submit_keeps_what_describes_the_work(gpu):
    """Right after the submits, every argument array the caller passed is overwritten (plans, sources, steps, ramps, text
    pointers and capacities, album descriptors, their page, plan and destination arrays) and every plan is destroyed, the
    plan cache cleared: the results are still those of the synchronous calls."""
    L = gpu.lib
    imgs = _images(7)
    plans = [gpu.plan(i.shape[1], i.shape[0], i.shape[2], api.Config(**kw), **rq) for i, (_, kw, rq) in zip(imgs, IO.CASES)]
    albums, gplans, _ = GA._mixed(gpu, np.random.default_rng(29))
    n = len(plans)
    want_b = gpu.batch_brightness(plans, imgs)
    want_t = gpu.batch_ascii(plans, imgs, ARGS)
    want_f = IO._frames(gpu, plans, imgs)
    want_a = GA._copy(gpu.gif_albums(albums))
    frames = [np.zeros_like(f) for f in want_f]
    jobs = api.HostJobs(plans, imgs, frames)
    P, S, SS = api._job_arrays(plans, imgs)
    b = np.zeros(n, np.float32)
    Pa, Sa, SSa, A, T, caps, texts = gpu._ascii_arrays(plans, imgs, ARGS)
    gjob = api.GifAlbumsJob(gpu, albums)
    tickets = [jobs.submit(gpu, 2)]
    for call in (lambda t: L.imp_gpu_batch_brightness_submit_host(n, P, S, SS, b.ctypes.data, 2, t),
                 lambda t: L.imp_gpu_batch_ascii_submit_host(n, Pa, Sa, SSa, A, T, caps, 2, t),
                 lambda t: L.imp_gpu_gif_albums_submit_host(gjob.arr, gjob.n, 2, t)):
        t = C.c_void_p()
        gpu.check(call(C.byref(t)))
        tickets.append(t)
    for arr in (jobs.P, jobs.S, jobs.D, P, S, Pa, Sa, T):
        C.memset(arr, 0, C.sizeof(arr))
    for arr in (jobs.SS, jobs.DS, SS, SSa, caps):
        C.memset(arr, 0xff, C.sizeof(arr))
    for i in range(n):
        A[i] = None if ARGS[i] else b"wide"                           # the other ramp
    for j in gjob.jobs:
        for arr in (j.arr, j.P, j.D, j.DS):
            C.memset(arr, 0, C.sizeof(arr))
    C.memset(gjob.arr, 0, C.sizeof(gjob.arr))
    for p in plans + gplans:
        p.close()
    gpu.plan_cache_clear()
    for t in tickets:
        _wait(gpu, t)
    assert all(np.array_equal(x, y) for x, y in zip(frames, want_f))
    assert b.tobytes() == want_b.tobytes()
    assert [x.tobytes() for x in texts] == want_t
    GA._assert_albums_equal(gjob.outs, want_a, "captured")


# A fresh process on two devices: the submits are made on device 1, the thread then moves to device 0 and waits. The
# results are exact, and device 0, whose context exists only from the switch on, received none of the work (no lane,
# staging or canvas memory appears there).
_DEVICES = r"""
import sys, ctypes as C, numpy as np
sys.path.insert(0, "."); sys.path.insert(0, "tests")
import ngx_http_imgproc_b200 as M
from ngx_http_imgproc_b200 import api
import test_gif_albums as GA, test_submit_host as T
cu = None
def free_bytes(ordinal):
    ctx, dev, free, total = C.c_void_p(), C.c_int(), C.c_size_t(), C.c_size_t()
    assert cu.cuDeviceGet(C.byref(dev), ordinal) == 0 and cu.cuDevicePrimaryCtxRetain(C.byref(ctx), dev) == 0
    assert cu.cuCtxPushCurrent_v2(ctx) == 0 and cu.cuMemGetInfo_v2(C.byref(free), C.byref(total)) == 0
    assert cu.cuCtxPopCurrent_v2(C.byref(ctx)) == 0 and cu.cuDevicePrimaryCtxRelease_v2(dev) == 0
    return free.value
def active(ordinal):
    dev, flags, on = C.c_int(), C.c_uint(), C.c_int()
    assert cu.cuDeviceGet(C.byref(dev), ordinal) == 0 and cu.cuDevicePrimaryCtxGetState(dev, C.byref(flags), C.byref(on)) == 0
    return bool(on.value)
L = M.library(); L.init(1)
cu = C.CDLL("libcuda.so.1"); assert cu.cuInit(0) == 0
assert active(1) and not active(0)
albums, gplans, _ = GA._mixed(L, np.random.default_rng(41))
imgs, plans = T._images(0), T._plans(L)
want_a = GA._copy(L.gif_albums(albums)); want_b = L.batch_brightness(plans, imgs)
job = api.GifAlbumsJob(L, albums)
tg = job.submit(L, 4)
tb, b = L.batch_brightness_submit(plans, imgs, 4)
L.set_device(0)
assert active(0)
before = free_bytes(0)
api.HostJobs.wait(L, tb); api.HostJobs.wait(L, tg)
GA._assert_albums_equal(job.outs, want_a, "device 1")
assert b.tobytes() == want_b.tobytes()
drop = before - free_bytes(0)
assert drop < (64 << 20), drop
print("DEVICES OK")
"""


@pytest.mark.gpu
def test_the_work_runs_on_the_device_current_at_the_submit():
    if M.library().device_count() < 2:
        pytest.skip("needs two or more GPUs")
    r = subprocess.run([sys.executable, "-c", _DEVICES], cwd=ROOT, capture_output=True, text=True, timeout=900,
                       env={k: v for k, v in os.environ.items() if k != "IMP_GPU_DEVICES"})
    assert r.returncode == 0 and "DEVICES OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


_DBG = r"""
import sys, ctypes as C, numpy as np
sys.path.insert(0, "."); sys.path.insert(0, "tests")
import ngx_http_imgproc_b200 as M
from ngx_http_imgproc_b200 import api
import test_gif_albums as GA
L = M.library(); L.init(0)
L.lib.imp_gpu_debug_flags.restype = C.c_uint
albums, plans, rqs = GA._mixed(L, np.random.default_rng(41))
want = GA._copy(L.gif_albums(albums))
job = api.GifAlbumsJob(L, albums)
api.HostJobs.wait(L, job.submit(L, 4))
GA._assert_albums_equal(job.outs, want, "debug build")
flags = L.lib.imp_gpu_debug_flags()
print("DBG", hex(flags))
assert flags == 0, hex(flags)
"""


@pytest.mark.gpu
def test_album_submit_on_the_debug_build():
    dbg = os.path.join(ROOT, "ngx_http_imgproc_b200", "libimp_gpu_dbg.so")
    assert os.path.exists(dbg), "the debug library is built by __graft_entry__.build()"
    r = subprocess.run([sys.executable, "-c", _DBG], cwd=ROOT, env=dict(os.environ, IMP_GPU_LIB=dbg), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "DBG 0x0" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]
