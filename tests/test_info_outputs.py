"""Brightness (format=json) and ASCII (format=text) answers of the host-batch path and of the operator layer, on a B200:
job i runs its plan exactly as imp_gpu_batch_run_host would, and only the answer comes back."""
import ctypes as C

import numpy as np
import pytest

import ngx_http_imgproc_b200 as M
from ngx_http_imgproc_b200 import api
from conftest import rnd_image, smooth_image
from test_planner_host import _oracle

pytestmark = pytest.mark.gpu

WM = rnd_image(7, 12, 20, 4)
WMKW = dict(allow_experiments=True, max_filters=8, watermark=WM, wm_gravity_x="r", wm_gravity_y="b", wm_offset_x=3, wm_offset_y=2, wm_opacity=60)
EXP = dict(allow_experiments=True, max_filters=8)

# (source shape, config, request): a strip pass, a gather-tile pass, cubic, sigma 2.3 and 6 blurs, a chain split into passes,
# rotate / flip, a watermark, flatten; 1-, 3- and 4-channel sources of odd sizes
CASES = [((121, 203, 3), dict(), dict(resize="67,40")),
         ((75, 97, 4), dict(), dict(resize="180,140,up", simple=True)),
         ((45, 61, 3), dict(), dict(resize="121,90,up")),
         ((99, 131, 3), EXP, dict(filters=["blur=2.3"])),
         ((67, 89, 4), EXP, dict(filters=["blur=6"])),
         ((83, 117, 3), EXP, dict(resize="77,51", filters=["blur=0.8", "rainbow=mid", "blur=1.5", "gradmap=306090,eecc00"])),
         ((57, 93, 1), EXP, dict(filters=["rotate=90", "flip=10"])),
         ((63, 101, 4), WMKW, dict(crop="81px,55px,c,c", filters=["modulate=0,0,100"])),
         ((53, 71, 4), dict(), dict(resize="35", flatten=True)),
         ((33, 47, 1), dict(), dict()),
         ((1, 37, 3), dict(), dict(filters=["gamma=1.3"])),
         ((29, 1, 4), dict(), dict(filters=["contrast=1.2"])),
         ((61, 79, 3), EXP, dict(filters=["blur=2.3", "vignette=0.8", "rotate=90"]))]


def _vignette(rq):
    return any("vignette" in f for f in rq.get("filters", []))


def _jobs(gpu, cases=CASES, seed=0):
    imgs = [smooth_image(seed + k, *shape) if k % 2 else rnd_image(seed + k, *shape) for k, (shape, _, _) in enumerate(cases)]
    plans = [gpu.plan(i.shape[1], i.shape[0], i.shape[2], api.Config(**kw), **rq) for i, (_, kw, rq) in zip(imgs, cases)]
    return imgs, plans


def _frames(gpu, plans, imgs):
    outs = [np.zeros((p.out_h, p.out_w, p.out_c), np.uint8) for p in plans]
    api.run_host_batch(gpu, plans, imgs, outs)
    return outs


def _numpy_brightness(frame):
    """The per-pixel expression in float64 over the frame, sum / (w*h) / 255."""
    f = frame.astype(np.int64)
    if f.shape[2] == 1:
        v = f[:, :, 0].astype(np.float64)
    else:
        b, g, r = f[:, :, 0], f[:, :, 1], f[:, :, 2]
        v = np.sqrt((r * r) * 0.241 + (g * g) * 0.691 + (b * b) * 0.068)
    return float(v.sum()) / (frame.shape[0] * frame.shape[1]) / 255.0


def _within_one_ulp(got, ref64):
    r = np.float32(ref64)
    return got in (r, np.nextafter(r, np.float32(np.inf)), np.nextafter(r, np.float32(-np.inf)))


def _pinned(gpu, arr, keep):
    p = C.c_void_p()
    gpu.check(gpu.lib.imp_gpu_host_alloc(C.byref(p), arr.nbytes))
    keep.append(p)
    out = np.ctypeslib.as_array((C.c_ubyte * arr.nbytes).from_address(p.value)).reshape(arr.shape)
    out[...] = arr
    return out


def _close(plans):
    for p in plans:
        p.close()


def test_mixed_batch_brightness_matches_the_frame_and_the_oracle(gpu, orc):
    imgs, plans = _jobs(gpu)
    frames = _frames(gpu, plans, imgs)
    got = gpu.batch_brightness(plans, imgs)
    o = orc.orc()
    for k, ((shape, kw, rq), img, fr) in enumerate(zip(CASES, imgs, frames)):
        assert _within_one_ulp(got[k], _numpy_brightness(fr)), (k, rq, got[k], _numpy_brightness(fr))
        code, _, ref_frame = _oracle(orc, img, rq, kw)
        assert code == 0
        ref = o.perceived_brightness(ref_frame)
        assert abs(float(got[k]) - ref) < 1e-4, (k, rq, got[k], ref)
        if abs((ref * 100) % 1 - 0.5) >= 0.01:
            assert round(float(got[k]) * 100) == round(ref * 100), (k, rq, got[k], ref)
    _close(plans)


def test_mixed_batch_ascii_matches_the_oracle(gpu, orc):
    imgs, plans = _jobs(gpu)
    frames = _frames(gpu, plans, imgs)
    args = ["wide" if k % 2 else None for k in range(len(CASES))]
    texts = gpu.batch_ascii(plans, imgs, args)
    o = orc.orc()
    for k, ((shape, kw, rq), img, fr) in enumerate(zip(CASES, imgs, frames)):
        assert len(texts[k]) == (fr.shape[1] + 1) * fr.shape[0] - 1
        if _vignette(rq):                                              # vignette parity with the oracle is <= 1 LSB
            assert texts[k] == gpu.ascii(fr, args[k] or ""), (k, rq)
        else:
            ref = _oracle(orc, img, rq, kw)[2]
            assert texts[k] == o.ascii(ref, args[k] == "wide"), (k, rq)
    _close(plans)


def test_brightness_bits_do_not_depend_on_the_batch(gpu):
    imgs, plans = _jobs(gpu)
    frames = _frames(gpu, plans, imgs)
    base = gpu.batch_brightness(plans, imgs, n_streams=4)
    for ns in (1, 8):
        assert gpu.batch_brightness(plans, imgs, n_streams=ns).tobytes() == base.tobytes()
    assert gpu.batch_brightness(plans, imgs).tobytes() == base.tobytes()                  # repeated
    assert gpu.batch_brightness(plans[::-1], imgs[::-1])[::-1].tobytes() == base.tobytes()  # other positions and neighbours
    extra_imgs, extra_plans = _jobs(gpu, seed=50)
    mixed = gpu.batch_brightness(extra_plans[:5] + plans + extra_plans[5:], extra_imgs[:5] + imgs + extra_imgs[5:], n_streams=2)
    assert mixed[5:5 + len(plans)].tobytes() == base.tobytes()
    for k, fr in enumerate(frames):                                   # the single-frame entry point on the materialised frame
        assert np.float32(gpu.brightness(fr)).tobytes() == base[k].tobytes(), k
    _close(plans + extra_plans)


def test_pinned_and_pageable_sources_at_full_size(gpu):
    keep = []
    try:
        img4 = rnd_image(21, 3000, 4000, 3)
        p4 = gpu.plan(4000, 3000, 3, api.Config(allow_experiments=True), filters=["blur=2.3", "vignette=0.8", "rotate=90"])
        wm = rnd_image(3, 64, 256, 4)
        cfg2 = api.Config(watermark=wm, wm_gravity_x="r", wm_gravity_y="b", wm_offset_x=10, wm_offset_y=10, wm_opacity=60)
        srcs2 = [rnd_image(30 + k, 2160, 3840, 4) for k in range(4)]
        p2 = gpu.plan(3840, 2160, 4, cfg2, crop="3600px,2025px,c,c", resize="800,450")
        plans = [p4] + [p2] * 16
        pageable = [img4] + [srcs2[k % 4] for k in range(16)]
        pin_pool = [_pinned(gpu, img4, keep)] + [_pinned(gpu, s, keep) for s in srcs2]
        pinned = [pin_pool[0]] + [pin_pool[1 + k % 4] for k in range(16)]
        frames = _frames(gpu, plans, pageable)
        b_page = gpu.batch_brightness(plans, pageable)
        b_pin = gpu.batch_brightness(plans, pinned)
        assert b_page.tobytes() == b_pin.tobytes()
        for k in (0, 1, 2, 3, 4):
            assert _within_one_ulp(b_page[k], _numpy_brightness(frames[k])), k
        t_page = gpu.batch_ascii(plans, pageable, "wide")
        t_pin = gpu.batch_ascii(plans, pinned, "wide")
        assert t_page == t_pin
        for k in (0, 1, 2, 3, 4):
            assert t_page[k] == gpu.ascii(frames[k], "wide"), k
        # pinned destinations take the direct copies
        out = _pinned(gpu, np.zeros(len(plans) * 4, np.uint8), keep).view(np.float32)
        P, S, SS = api._job_arrays(plans, pinned)
        gpu.check(gpu.lib.imp_gpu_batch_brightness_host(len(plans), P, S, SS, out.ctypes.data, 4))
        assert out.tobytes() == b_page.tobytes()
        p4.close(); p2.close()
    finally:
        for p in keep:
            gpu.lib.imp_gpu_host_free(p)


def test_one_more_launch_than_the_frame_path(gpu):
    cases = CASES[:3] + CASES[6:8]
    imgs, plans = _jobs(gpu, cases)
    outs = [np.zeros((p.out_h, p.out_w, p.out_c), np.uint8) for p in plans]
    assert sum(i.nbytes for i in imgs) + sum(o.nbytes for o in outs) < 4 << 20
    api.run_host_batch(gpu, plans, imgs, outs, n_streams=1)           # plans uploaded, lanes allocated
    l0 = gpu.launch_count()
    api.run_host_batch(gpu, plans, imgs, outs, n_streams=1)
    frame_launches = gpu.launch_count() - l0
    l0 = gpu.launch_count()
    gpu.batch_brightness(plans, imgs, n_streams=1)
    assert gpu.launch_count() - l0 == frame_launches + 1
    l0 = gpu.launch_count()
    gpu.batch_ascii(plans, imgs, "wide", n_streams=1)
    assert gpu.launch_count() - l0 == frame_launches + 1
    _close(plans)


def test_argument_errors_write_nothing(gpu):
    imgs, plans = _jobs(gpu, CASES[:2])
    packed = gpu.plan(imgs[0].shape[1], imgs[0].shape[0], 3, resize="40,30", pack=24)
    L = gpu.lib
    P, S, SS = api._job_arrays(plans, imgs)
    b = np.full(2, -7.0, np.float32)
    lens = [L.imp_gpu_ascii_length(p.out_w, p.out_h) for p in plans]
    bufs = [C.create_string_buffer(b"\x5a" * k, k) for k in lens]
    T = (C.c_void_p * 2)(*[C.addressof(x) for x in bufs])
    A = (C.c_char_p * 2)(None, b"wide")
    caps = (C.c_long * 2)(*lens)
    small = (C.c_long * 2)(lens[0], lens[1] - 1)
    bad = M.IMP_ERROR_INVALID_ARGS
    assert L.imp_gpu_batch_brightness_host(2, None, S, SS, b.ctypes.data, 4) == bad
    assert L.imp_gpu_batch_brightness_host(2, P, S, None, b.ctypes.data, 4) == bad
    assert L.imp_gpu_batch_brightness_host(2, P, S, SS, None, 4) == bad
    assert L.imp_gpu_batch_ascii_host(2, P, S, SS, None, T, caps, 4) == bad
    assert L.imp_gpu_batch_ascii_host(2, P, S, SS, A, T, None, 4) == bad
    assert L.imp_gpu_batch_ascii_host(2, P, S, SS, A, T, small, 4) == bad
    Pp, Sp, SSp = api._job_arrays([plans[0], packed], [imgs[0], imgs[0]])
    assert L.imp_gpu_batch_brightness_host(2, Pp, Sp, SSp, b.ctypes.data, 4) == bad
    assert L.imp_gpu_batch_ascii_host(2, Pp, Sp, SSp, A, T, caps, 4) == bad
    assert (b == -7.0).all() and all(x.raw == b"\x5a" * k for x, k in zip(bufs, lens))
    assert L.imp_gpu_batch_brightness_host(0, P, S, SS, b.ctypes.data, 4) == M.IMP_OK and (b == -7.0).all()
    _close(plans + [packed])


def test_operators_answer_what_the_flush_would_leave(gpu):
    ops = api.OpsLayer(gpu)
    L = gpu.lib
    for (shape, kw, rq) in (CASES[0], CASES[6], CASES[7], CASES[8]):
        img = rnd_image(sum(shape), *shape)
        cfg = api.Config(**kw)
        plan = gpu.plan(shape[1], shape[0], shape[2], cfg, **rq)
        want_b = gpu.batch_brightness([plan], [img])[0]
        want_t = gpu.batch_ascii([plan], [img], "wide")[0]
        frame = _frames(gpu, [plan], [img])[0]
        plan.close()
        req = dict(crop=rq.get("crop"), resize=rq.get("resize"), filters=rq.get("filters", ()), simple=rq.get("simple", False),
                   flatten=rq.get("flatten", False))
        code, ptrs = ops.record([img], cfg, **req)
        assert code == 0
        p = ptrs[0]
        pending = L.imp_ops_pending(p)
        v = C.c_float()
        assert L.imp_Brightness(p, C.byref(v)) == 0 and np.float32(v.value).tobytes() == want_b.tobytes(), rq
        n = len(want_t)
        buf = C.create_string_buffer(n)
        assert L.imp_Ascii(p, b"wide", buf, n) == 0 and buf.raw[:n] == want_t, rq
        assert L.imp_Ascii(p, b"wide", buf, n - 1) == M.IMP_ERROR_INVALID_ARGS
        assert L.imp_ops_pending(p) == pending
        arr = (C.POINTER(api.IplImage) * 1)(p)
        assert L.imp_FlushAll(arr, 1) == 0
        im = arr[0].contents
        raw = (C.c_ubyte * (im.widthStep * im.height)).from_address(im.imageData)
        got = np.frombuffer(raw, np.uint8).reshape(im.height, im.widthStep)[:, :im.width * im.nChannels].reshape(im.height, im.width, im.nChannels)
        assert np.array_equal(got, frame), rq
        assert ops.brightness([img], cfg, **req) == (0, [float(want_b)])
        assert ops.ascii([img], cfg, "wide", **req) == (0, [want_t])


def test_idle_gray_frame_is_answered_as_bgr(gpu):
    ops = api.OpsLayer(gpu)
    img = rnd_image(9, 21, 34, 1)
    bgr = np.repeat(img, 3, axis=2)
    code, b = ops.brightness([img], api.Config())
    assert code == 0 and np.float32(b[0]).tobytes() == np.float32(gpu.brightness(bgr)).tobytes()
    code, t = ops.ascii([img], api.Config(), "wide")
    assert code == 0 and t[0] == gpu.ascii(bgr, "wide")
    img3 = rnd_image(10, 21, 34, 3)                                   # idle 3-channel: the frame as it is
    assert ops.brightness([img3], api.Config())[1][0] == gpu.brightness(img3)
