"""GPU parity tests (run on a real B200 with -m gpu). Everything goes through the C ABI of
libimp_gpu.so (ngx_http_imgproc_b200.api is a thin ctypes binding) and is compared with the oracle:
bit-exact everywhere except Vignette, where CUDA's and glibc's double-precision cos may differ in the
last ulp (tolerance 1 LSB, and the mismatch count must stay tiny)."""
import ctypes as C

import numpy as np
import pytest

import golden_util as G
from conftest import rnd_image, smooth_image
from ngx_http_imgproc_b200 import api
from test_planner_host import REQS, _oracle

pytestmark = pytest.mark.gpu


def _gpu_run(gpu, img, cfgkw, rq):
    code, step, plan = gpu.try_plan(img.shape[1], img.shape[0], img.shape[2], api.Config(**cfgkw), **rq)
    if code:
        return code, step, None
    try:
        return 0, step, plan.run_host(img)
    finally:
        plan.close()


def _assert_same(out, ref, rq, vig):
    """Bit-exact. vig: False, or (source shape, config kwargs, request) of a request with vignette ops, which is exact
    except at output pixels an ambiguous mask entry reaches (golden_util.assert_vignette_exact)."""
    if vig:
        G.assert_vignette_exact(out, ref, *vig, rq)
        return
    assert out.shape == ref.shape, (rq, out.shape, ref.shape)
    d = np.abs(out.astype(int) - ref.astype(int))
    assert d.max() == 0, (rq, int(d.max()), int((d > 0).sum()), d.size)


def _has_vignette(rq):
    return any("vignette" in f for f in rq.get("filters", []) or [])


def _vig(shape, kw, rq):
    """The vig argument of _assert_same for a request on a source of that shape."""
    return (shape, kw, rq) if _has_vignette(rq) else False


def test_kernels_actually_launch(gpu):
    before = gpu.launch_count()
    out = gpu.run(rnd_image(0, 16, 16, 3), resize="8,8")
    assert out.shape == (8, 8, 3) and gpu.launch_count() > before


@pytest.mark.parametrize("case", G.load(), ids=lambda c: c["name"])
def test_golden_vectors(gpu, case):
    """Vectors produced by the reference's own code + cv2 in the build container."""
    req = G.split_query(case["query"])
    code, step, out = _gpu_run(gpu, case["img"], case["cfgkw"], req)
    assert code == case["code"]
    if code:
        return
    _assert_same(out, case["out"], case["query"], _vig(case["img"].shape, case["cfgkw"], req))


def test_request_matrix_vs_oracle(gpu, orc):
    wm, wm3 = rnd_image(7, 12, 20, 4), rnd_image(8, 7, 9, 3)
    cfgkws = [dict(),
              dict(allow_experiments=True, max_filters=8, watermark=wm, wm_gravity_x="r", wm_gravity_y="b", wm_offset_x=3, wm_offset_y=2, wm_opacity=60),
              dict(allow_experiments=True, watermark=wm3, wm_gravity_x="c", wm_gravity_y="c", wm_offset_x=-4, wm_offset_y=5, wm_opacity=100),
              dict(max_w=100, max_h=50, watermark=wm, wm_gravity_x="l", wm_gravity_y="t", wm_offset_x=-5, wm_offset_y=-3, wm_opacity=37)]
    n = 0
    for ci, kw in enumerate(cfgkws):
        for (h, w, c) in [(60, 80, 3), (45, 64, 4), (33, 47, 1), (48, 64, 3)]:
            img = rnd_image(100 + ci, h, w, c) if ci % 2 == 0 else smooth_image(100 + ci, h, w, c)
            for rq in REQS:
                code, step, out = _gpu_run(gpu, img, kw, rq)
                c2, s2, o2 = _oracle(orc, img, rq, kw)
                assert code == c2 and (not code or step == s2), (ci, rq)
                if not code:
                    _assert_same(out, o2, (ci, (h, w, c), rq), _vig(img.shape, kw, rq))
                n += 1
    assert n > 800


FILTERS = ["flip=10", "flip=01", "flip=11", "rotate=90", "rotate=180", "rotate=270", "modulate=0,0,100", "modulate=60,70,80",
           "modulate=100,500,500", "modulate=180,-50,100", "colorize=704214,0.6", "colorize=ff0000", "gamma=1.3", "gamma=0.5",
           "contrast=1.5", "contrast=0.5", "contrast=3.7", "gradmap=306090,eecc00", "gradmap=000000,ff0000,ffffff", "vignette=0.8",
           "vignette=4,3", "vignette=0.5,0.7", "gotham=1", "lomo=1", "kelvin=1", "rainbow=full", "rainbow=mid", "rainbow=pale",
           "scanline=0", "scanline=0.5,0.25,1,1", "scanline=0.3,0.9,2,3", "blur=0.5", "blur=1", "blur=2.3", "blur=6"]


@pytest.mark.parametrize("f", FILTERS)
def test_each_filter_all_byte_values(gpu, orc, f):
    """Every filter on an image holding all 2^24 BGR triples' worth of variety: a 256x256 ramp grid + noise,
    3- and 4-channel, odd sizes so that widthStep != w*C."""
    kw = dict(allow_experiments=True)
    b, g = np.mgrid[0:256, 0:256].astype(np.uint8)
    for c in (3, 4):
        img = np.zeros((256, 256, c), np.uint8)
        img[:, :, 0], img[:, :, 1] = b, g
        img[:, :, 2] = rnd_image(1, 256, 256, 1)[:, :, 0]
        if c == 4:
            img[:, :, 3] = rnd_image(2, 256, 256, 1)[:, :, 0]
        for im in (img, rnd_image(5, 131, 67, c)):
            code, _, out = _gpu_run(gpu, im, kw, dict(filters=[f]))
            c2, _, o2 = _oracle(orc, im, dict(filters=[f]), kw)
            assert code == c2 == 0
            _assert_same(out, o2, f, _vig(im.shape, kw, dict(filters=[f])))


def test_resize_fuzz_vs_oracle(gpu, orc):
    """Random size pairs for every interpolation the path has (NN, AREA int/frac, CUBIC, LINEAR)."""
    rng = np.random.default_rng(42)
    cfg = dict(max_w=0, max_h=0)
    for it in range(150):
        sw, sh = int(rng.integers(1, 200)), int(rng.integers(1, 150))
        dw, dh = int(rng.integers(1, 260)), int(rng.integers(1, 200))
        c = int(rng.choice([1, 3, 4]))
        img = rng.integers(0, 256, (sh, sw, c), dtype=np.uint8)
        for rq in (dict(resize=f"{dw},{dh},up"), dict(resize=f"{dw},{dh},up", simple=True), dict(resize=f"{dw},{dh},up", interp=1), dict(resize=f"{dw},{dh}")):
            code, _, out = _gpu_run(gpu, img, cfg, rq)
            c2, _, o2 = _oracle(orc, img, rq, cfg)
            assert code == c2 == 0, rq
            _assert_same(out, o2, (sw, sh, c, rq), False)


def test_edge_shapes(gpu, orc):
    kw = dict(allow_experiments=True, max_filters=8)
    for (h, w, c) in [(1, 1, 3), (1, 1, 4), (1, 7, 1), (9, 1, 4), (2, 3, 3), (8, 32, 4), (9, 33, 3), (257, 3, 3)]:
        img = rnd_image(h * 31 + w, h, w, c)
        for rq in [dict(), dict(filters=["blur=2.3"]), dict(filters=["blur=12"]), dict(resize="5,4,up"), dict(resize="1,1"),
                   dict(filters=["rotate=90", "vignette=0.8", "blur=1"]), dict(filters=["gotham=1", "rotate=270"]), dict(flatten=True)]:
            code, _, out = _gpu_run(gpu, img, kw, rq)
            c2, _, o2 = _oracle(orc, img, rq, kw)
            assert code == c2, ((h, w, c), rq)
            if not code:
                _assert_same(out, o2, ((h, w, c), rq), _vig(img.shape, kw, rq))
    for v in (0, 255):
        img = np.full((40, 50, 4), v, np.uint8)
        for rq in [dict(filters=["kelvin=1"]), dict(resize="20,13"), dict(flatten=True), dict(filters=["modulate=90,200,50"])]:
            _, _, out = _gpu_run(gpu, img, kw, rq)
            _assert_same(out, _oracle(orc, img, rq, kw)[2], rq, False)


# ---- the five BASELINE.json configurations ------------------------------------------------------------------
def test_cfg1_1080p_to_640x360(gpu, orc):
    img = rnd_image(1, 1080, 1920, 3)
    for rq in (dict(resize="640,360"), dict(resize="640,360", interp=1)):
        out = _gpu_run(gpu, img, {}, rq)[2]
        _assert_same(out, _oracle(orc, img, rq, {})[2], rq, False)


def test_cfg2_4k_crop_area_watermark_full_size(gpu, orc):
    img = smooth_image(2, 2160, 3840, 4)
    wm = rnd_image(3, 64, 256, 4)
    wm[:, :, 3] = np.linspace(0, 255, 256).astype(np.uint8)[None, :]
    kw = dict(watermark=wm, wm_gravity_x="r", wm_gravity_y="b", wm_offset_x=10, wm_offset_y=10, wm_opacity=60)
    rq = dict(crop="3600px,2025px,c,c", resize="800,450")
    out = _gpu_run(gpu, img, kw, rq)[2]
    assert out.shape == (450, 800, 4)
    _assert_same(out, _oracle(orc, img, rq, kw)[2], rq, False)


def test_cfg3_gif_frames_cubic_sepia_batched(gpu, orc):
    """200 frames 480x270x4 -> cubic 2x + sepia as ONE batch launch; every frame checked."""
    base = smooth_image(4, 270, 480, 4)
    base[:, :, 3] = np.where(base[:, :, 3] > 127, 255, 0)
    frames = [np.roll(base, (i, 2 * i), (0, 1)) for i in range(200)]
    rq = dict(resize="960,540,up", filters=["modulate=0,0,100", "colorize=704214,0.6"])
    outs = _device_batch(gpu, frames, [rq] * 200, {})
    for i in (0, 1, 57, 199):
        _assert_same(outs[i], _oracle(orc, frames[i], rq, {})[2], (i, rq), False)
    nn = dict(resize="960,540,up", simple=True, filters=rq["filters"])
    _assert_same(_gpu_run(gpu, frames[3], {}, nn)[2], _oracle(orc, frames[3], nn, {})[2], nn, False)


def test_cfg4_12mp_blur_vignette_rotate_full_size(gpu, orc):
    img = smooth_image(5, 3000, 4000, 3)
    kw = dict(allow_experiments=True)
    rq = dict(filters=["blur=2.3", "vignette=0.8", "rotate=90"])
    out = _gpu_run(gpu, img, kw, rq)[2]
    assert out.shape == (4000, 3000, 3)
    _assert_same(out, _oracle(orc, img, rq, kw)[2], rq, _vig(img.shape, kw, rq))


def test_cfg5_thumbnail_farm_sample(gpu, orc):
    """Mixed-size sources -> 256x256 + watermark in one batch (sizes as in SURVEY §8d cfg5, 24 jobs)."""
    rng = np.random.default_rng(6)
    wm = rnd_image(61, 64, 64, 4)
    kw = dict(max_w=0, max_h=0, watermark=wm, wm_gravity_x="r", wm_gravity_y="b", wm_offset_x=8, wm_offset_y=8, wm_opacity=100)
    imgs, rqs = [], []
    for i in range(24):
        w, h = int(rng.integers(320, 2049)), int(rng.integers(240, 1537))
        c = 3 if rng.random() < 0.75 else 4
        imgs.append(rnd_image(600 + i, h, w, c))
        rqs.append(dict(resize="256,256"))
    imgs.append(rnd_image(700, 512, 1024, 3)); rqs.append(dict(resize="256,256"))      # integer 4x2
    outs = _device_batch(gpu, imgs, rqs, kw)
    for i in range(len(imgs)):
        _assert_same(outs[i], _oracle(orc, imgs[i], rqs[i], kw)[2], (i, imgs[i].shape), False)


# ---- batch / farm API ------------------------------------------------------------------------------------------
def _device_batch(gpu, imgs, rqs, cfgkw):
    """imp_gpu_batch_* over device-resident frames (uploads with the ABI's own helpers)."""
    L = gpu.lib
    plans, bufs, outs = [], [], []
    batch = api.Batch(gpu)
    for img, rq in zip(imgs, rqs):
        img = np.ascontiguousarray(img)
        p = gpu.plan(img.shape[1], img.shape[0], img.shape[2], api.Config(**cfgkw), **rq)
        d_in, d_out, pi, po = C.c_void_p(), C.c_void_p(), C.c_int(), C.c_int()
        gpu.check(L.imp_gpu_malloc_pitch(C.byref(d_in), C.byref(pi), img.shape[1] * img.shape[2], img.shape[0]))
        gpu.check(L.imp_gpu_malloc_pitch(C.byref(d_out), C.byref(po), p.out_w * p.out_c, p.out_h))
        gpu.check(L.imp_gpu_upload_2d(d_in, pi.value, img.ctypes.data, img.strides[0], img.shape[1] * img.shape[2], img.shape[0], None))
        batch.add(p, d_in.value, pi.value, d_out.value, po.value)
        plans.append(p); bufs.append((d_in, d_out, po.value))
    gpu.check(L.imp_gpu_sync(None))
    before = gpu.launch_count()
    batch.launch()
    gpu.check(L.imp_gpu_sync(None))
    assert gpu.launch_count() - before == batch.launches_per_run
    for p, (d_in, d_out, po) in zip(plans, bufs):
        out = np.empty((p.out_h, p.out_w, p.out_c), np.uint8)
        gpu.check(L.imp_gpu_download_2d(out.ctypes.data, out.strides[0], d_out, po, p.out_w * p.out_c, p.out_h, None))
        outs.append(out)
    gpu.check(L.imp_gpu_sync(None))
    for p, (d_in, d_out, po) in zip(plans, bufs):
        L.imp_gpu_free(d_in); L.imp_gpu_free(d_out); p.close()
    batch.close()
    return outs


def test_batch_mixed_plans_one_launch_per_variant(gpu, orc):
    kw = dict(allow_experiments=True, max_filters=8)
    rqs = [dict(resize="40,30"), dict(resize="41,29"), dict(filters=["blur=1.5", "gamma=1.2"]), dict(resize="100,90,up"),
           dict(filters=["rotate=90"]), dict(resize="20,20", filters=["blur=2", "kelvin=1", "blur=0.7"]), dict(crop="30px,30px,c,c", resize="17,19")]
    imgs = [rnd_image(i, 50 + i, 60 + 2 * i, 3 if i % 2 else 4) for i in range(len(rqs))]
    outs = _device_batch(gpu, imgs, rqs, kw)
    for img, rq, out in zip(imgs, rqs, outs):
        _assert_same(out, _oracle(orc, img, rq, kw)[2], rq, False)


def test_run_device_matches_oracle(gpu, orc):
    """imp_gpu_run_device: one frame in device buffers through the batch's launch steps, every job passed by value and the
    scratch allocated on the stream. A strip pass (cfg2's request, reduced), a gather tile pass, a multi-pass chain through
    scratch, a blur beyond the tile kernel's radius (two launches through the u16 plane) and a source whose pitch is not a
    multiple of 16 (a pass-0 blur then takes the two-launch path as well)."""
    L = gpu.lib
    kw = dict(allow_experiments=True, max_filters=8)
    kw_wm = dict(kw, watermark=rnd_image(3, 16, 64, 4), wm_gravity_x="r", wm_gravity_y="b", wm_offset_x=10, wm_offset_y=10, wm_opacity=60)
    cases = [(smooth_image(1, 540, 960, 4), kw_wm, dict(crop="900px,506px,c,c", resize="200,112"), 0),
             (smooth_image(2, 300, 400, 3), kw, dict(filters=["rotate=90"]), 0),
             (smooth_image(3, 120, 160, 3), kw, dict(resize="100,75", filters=["blur=2", "kelvin=1", "blur=0.7"]), 0),
             (smooth_image(4, 120, 160, 4), kw, dict(filters=["blur=6"]), 0),
             (smooth_image(5, 135, 240, 3), kw, dict(filters=["blur=2.3", "gamma=1.2"]), 5)]
    for img, cfgkw, rq, pad in cases:
        h, w, c = img.shape
        p = gpu.plan(w, h, c, api.Config(**cfgkw), **rq)
        d_in, d_out, pi, po = C.c_void_p(), C.c_void_p(), C.c_int(), C.c_int()
        if pad:
            sp = w * c + pad
            gpu.check(L.imp_gpu_malloc_pitch(C.byref(d_in), C.byref(pi), sp * h, 1))
        else:
            gpu.check(L.imp_gpu_malloc_pitch(C.byref(d_in), C.byref(pi), w * c, h))
            sp = pi.value
        gpu.check(L.imp_gpu_malloc_pitch(C.byref(d_out), C.byref(po), p.out_w * p.out_c, p.out_h))
        gpu.check(L.imp_gpu_upload_2d(d_in, sp, img.ctypes.data, img.strides[0], w * c, h, None))
        before = gpu.launch_count()
        p.run_device(d_in.value, sp, d_out.value, po.value)
        out = np.empty((p.out_h, p.out_w, p.out_c), np.uint8)
        gpu.check(L.imp_gpu_download_2d(out.ctypes.data, out.strides[0], d_out, po.value, p.out_w * p.out_c, p.out_h, None))
        gpu.check(L.imp_gpu_sync(None))
        assert gpu.launch_count() - before >= p.passes, rq
        L.imp_gpu_free(d_in); L.imp_gpu_free(d_out); p.close()
        _assert_same(out, _oracle(orc, img, rq, cfgkw)[2], rq, False)


def test_host_batch_and_farm_match_single_runs(gpu, orc):
    kw = dict(max_w=0, max_h=0)
    imgs = [smooth_image(i, 300 + 7 * i, 400 + 5 * i, 3 if i % 3 else 4) for i in range(9)]
    rq = dict(crop="1,1", resize="128,128", filters=["gamma=1.1"])
    plans = [gpu.plan(im.shape[1], im.shape[0], im.shape[2], api.Config(**kw), **rq) for im in imgs]
    dsts = [np.zeros((p.out_h, p.out_w, p.out_c), np.uint8) for p in plans]
    api.run_host_batch(gpu, plans, imgs, dsts, n_streams=3)
    for im, d in zip(imgs, dsts):
        _assert_same(d, _oracle(orc, im, rq, kw)[2], rq, False)
    n_gpus = min(2, gpu.device_count())
    dsts2 = [np.zeros_like(d) for d in dsts]
    api.run_host_batch(gpu, plans, imgs, dsts2, n_streams=2, n_gpus=n_gpus)
    for a, b in zip(dsts, dsts2):
        assert np.array_equal(a, b)
    for p in plans:
        p.close()


# ---- size-independent properties at full sizes --------------------------------------------------------------------
def test_properties_full_size(gpu):
    img = rnd_image(9, 3000, 4000, 3)
    r = img
    for _ in range(4):
        r = gpu.run(r, filters=["rotate=90"])
    assert np.array_equal(r, img)                                             # four quarter turns = identity
    assert np.array_equal(gpu.run(gpu.run(img, filters=["flip=11"]), filters=["rotate=180"]), img)
    assert np.array_equal(gpu.run(img, filters=["rotate=90"]), np.ascontiguousarray(np.rot90(img, -1)))
    assert np.array_equal(gpu.run(img, crop="1000px,700px,37px,91px"), img[91:791, 37:1037])
    a = gpu.run(img, crop="3000px,2000px,c,c", resize="750,500")
    b = gpu.run(np.ascontiguousarray(img[500:2500, 500:3500]), resize="750,500")
    assert np.array_equal(a, b)                                               # crop folded into the gather == crop then resize
    c1 = gpu.run(img, filters=["blur=2.3", "rotate=90"])
    c2 = gpu.run(gpu.run(img, filters=["rotate=90"]), filters=["blur=2.3"])
    assert np.array_equal(c1, c2)                                             # blur commutes with the dihedral maps
    flat = np.full((1500, 2000, 4), 77, np.uint8)
    assert (gpu.run(flat, resize="333,211") == 77).all() and (gpu.run(flat, filters=["blur=6"]) == 77).all()


def test_perceived_brightness_reduction(gpu, orc):
    """SURVEY 8f-1: Info()'s brightness. The reference's sequential float32 sum is order-dependent, so parity is the
    JSON integer round(brightness*100) and a 1e-4 absolute band on the value itself."""
    o = orc.orc()
    for (h, w, c) in [(2, 4, 3), (270, 480, 4), (1080, 1920, 3), (33, 47, 1), (1, 1, 3)]:
        img = smooth_image(h + w, h, w, c) if h > 2 else np.array([[[0,0,0],[255,255,255],[10,128,250],[200,30,180]],[[37,201,99],[128,128,128],[255,0,170],[3,2,1]]], np.uint8)
        got, ref = gpu.brightness(img), o.perceived_brightness(img)
        assert abs(got - ref) < 1e-4, (h, w, c, got, ref)
        if abs(ref * 100 - round(ref * 100)) < 0.49:
            assert round(got * 100) == round(ref * 100)
    assert abs(gpu.brightness(np.array([[[0,0,0],[255,255,255],[10,128,250],[200,30,180]],[[37,201,99],[128,128,128],[255,0,170],[3,2,1]]], np.uint8)) - 0.45781034) < 1e-6   # App. B


def test_direct_fallback_kernels_subprocess(orc):
    """The general direct-from-global kernels (taken for unaligned pitches, oversized footprints, sigma > 4) stay
    parity-green: the same request matrix in a child process with IMP_GPU_FORCE_DIRECT=1."""
    import os, subprocess, sys
    code = r"""
import sys, numpy as np
sys.path.insert(0, "."); sys.path.insert(0, "tests")
import ngx_http_imgproc_b200 as M
from ngx_http_imgproc_b200 import api
from oracle import oracle as O
from conftest import rnd_image, smooth_image
from test_planner_host import REQS, _oracle
from test_gpu_parity import _gpu_run, _assert_same, _vig
L = M.library(); L.init(0)
wm = rnd_image(7, 12, 20, 4)
kw = dict(allow_experiments=True, max_filters=8, watermark=wm, wm_gravity_x="r", wm_gravity_y="b", wm_offset_x=3, wm_offset_y=2, wm_opacity=60)
n = 0
for (h, w, c) in [(60, 80, 3), (45, 64, 4), (33, 47, 1)]:
    img = smooth_image(h, h, w, c)
    for rq in REQS + [dict(resize="20,15"), dict(resize="27,31"), dict(filters=["blur=2.3", "rotate=90"]), dict(filters=["blur=6"])]:
        code, step, out = _gpu_run(L, img, kw, rq)
        c2, s2, o2 = _oracle(O, img, rq, kw)
        assert code == c2, rq
        if not code:
            _assert_same(out, o2, rq, _vig(img.shape, kw, rq))
        n += 1
img = rnd_image(1, 540, 960, 3)
for rq in (dict(resize="320,180"), dict(resize="213,120"), dict(resize="1500,900,up"), dict(filters=["blur=2.3"])):
    _assert_same(_gpu_run(L, img, dict(max_w=0, max_h=0), rq)[2], _oracle(O, img, rq, dict(max_w=0, max_h=0))[2], rq, False)
print("DIRECT_OK", n)
"""
    env = dict(os.environ, IMP_GPU_FORCE_DIRECT="1")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    assert "DIRECT_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]


def test_ascii_and_encoder_packing(gpu, orc):
    """SURVEY 8f-3/8f-4: IplToFI24/32 packing folded into the store, and ASCII on the device."""
    o = orc.orc()
    ramp = np.arange(256, dtype=np.uint8).reshape(1, 256, 1).repeat(3, 2)
    for img in (ramp, smooth_image(3, 37, 53, 3), smooth_image(4, 64, 96, 4), rnd_image(5, 1, 1, 3)):
        for args, wide in (("wide", True), ("", False)):
            assert gpu.ascii(img, args) == o.ascii(img, wide)
    kw = dict(allow_experiments=True)
    for c in (3, 4, 1):
        img = smooth_image(20 + c, 90, 120, c)
        for rq in (dict(resize="45,37", pack=24), dict(resize="45,37", pack=32), dict(filters=["rotate=90", "blur=1.2", "vignette=0.6"], pack=32),
                   dict(crop="1,1", resize="200,200,up", filters=["flip=10"], pack=24, flatten=True)):
            code, _, out = _gpu_run(gpu, img, kw, rq)
            c2, _, ref = _oracle(orc, img, rq, kw)
            assert code == c2 == 0
            _assert_same(out, ref, rq, _vig(img.shape, kw, rq))


def test_gif_canvas_expansion(gpu, orc):
    """SURVEY 8f-2: palette-index frames + disposal replay -> BGRA canvases, against the restatement of
    advancedio.c:195-248 (itself pinned to the reference's LoadGIF in tests/test_oracle.py)."""
    rng = np.random.default_rng(11)
    o = orc.orc()
    for destructive in (False, True):
        for (cw, ch, n) in [(48, 27, 6), (131, 77, 9), (1, 1, 2)]:
            frames = []
            for f in range(n):
                w = cw if f == 0 else int(rng.integers(1, cw + 1)); h = ch if f == 0 else int(rng.integers(1, ch + 1))
                pitch = (w + 3) & ~3
                idx = rng.integers(0, 16, (h, pitch), dtype=np.uint8)
                frames.append(dict(indices=idx[:, :w] if pitch == w else np.ascontiguousarray(idx)[:, :w], left=0 if f == 0 else int(rng.integers(0, cw - w + 1)),
                                   top=0 if f == 0 else int(rng.integers(0, ch - h + 1)), dispose=int(rng.integers(0, 4)),
                                   key=int(rng.choice([-1, 0, 3, 7])), palette=rng.integers(0, 256, (256, 4), dtype=np.uint8)))
            for fr in frames:
                fr["indices"] = np.ascontiguousarray(fr["indices"])
            got = gpu.gif_expand(frames, cw, ch, destructive)
            ref = o.gif_expand(frames, cw, ch, destructive)
            for a, b in zip(got, ref):
                assert np.array_equal(a, b)


def _random_gif(rng, cw, ch, n):
    frames = []
    for f in range(n):
        w = cw if f == 0 else int(rng.integers(1, cw + 1)); h = ch if f == 0 else int(rng.integers(1, ch + 1))
        frames.append(dict(indices=np.ascontiguousarray(rng.integers(0, 16, (h, w), dtype=np.uint8)), left=0 if f == 0 else int(rng.integers(0, cw - w + 1)),
                           top=0 if f == 0 else int(rng.integers(0, ch - h + 1)), dispose=int(rng.integers(0, 4)),
                           key=int(rng.choice([-1, 0, 3, 7])), palette=rng.integers(0, 256, (256, 4), dtype=np.uint8)))
    return frames


def test_gif_album_pages_to_results_on_the_device(gpu, orc):
    """A whole GIF request through imp_gpu_gif_album_run_host: pages up as indices, canvases expanded on the device, the
    frame loop (bridge.c:576-656) over them — against the restatement of LoadGIF's loop followed by the oracle's chain on
    every canvas. Frame counts on both sides of the chunking, one launch group per chunk."""
    rng = np.random.default_rng(23)
    o = orc.orc()
    cases = [((48, 27, 5), dict(resize="96,54", simple=True), True),
             ((131, 77, 9), dict(crop="100px,60px,c,c", resize="50", filters=["modulate=0,0,100", "colorize=704214,0.6", "rotate=90"]), False),
             ((64, 64, 40), dict(resize="128,128,up", filters=["gamma=1.3"]), True),
             ((33, 21, 3), dict(), True)]
    for (cw, ch, n), rq, destructive in cases:
        frames = _random_gif(rng, cw, ch, n)
        canvases = o.gif_expand(frames, cw, ch, destructive)
        code, step, plan = gpu.try_plan(cw, ch, 4, api.Config(), **rq)
        assert code == 0
        try:
            before = gpu.launch_count()
            outs = gpu.gif_album(frames, cw, ch, destructive, plan)
            launches = gpu.launch_count() - before
        finally:
            plan.close()
        assert launches <= 1 + 4 * plan.passes + 4, (n, launches)      # expansion + one grouped launch per lane chunk and pass
        for k, (got, canvas) in enumerate(zip(outs, canvases)):
            c2, _, ref = _oracle(orc, canvas, rq, {})
            assert c2 == 0
            _assert_same(got, ref, (rq, k), False)


def test_gif_album_rejects_mismatched_plans(gpu):
    rng = np.random.default_rng(5)
    frames = _random_gif(rng, 40, 30, 2)
    code, _, plan = gpu.try_plan(41, 30, 4, api.Config(), resize="20")
    assert code == 0
    try:
        with pytest.raises(Exception):
            gpu.gif_album(frames, 40, 30, True, plan)
    finally:
        plan.close()


def test_ops_layer_gif_flush(gpu, orc):
    """imp_FlushAllGif: the operators are recorded on canvas-sized placeholder frames (LoadGIF still creates them), the flush
    takes its pixels from the pages. Same results as the host-canvas flush and as the oracle; frames with nothing recorded
    receive their canvas."""
    rng = np.random.default_rng(31)
    o = orc.orc()
    ops = api.OpsLayer(gpu)
    cw, ch, n = 90, 52, 7
    frames = _random_gif(rng, cw, ch, n)
    canvases = o.gif_expand(frames, cw, ch, True)
    for kw in (dict(resize="45,26", simple=True, filters=["flip=10"]), dict(crop="60px,40px,l,t", filters=["contrast=1.2"]), dict()):
        place = [np.full((ch, cw, 4), 0xEE, np.uint8) for _ in range(n)]              # never read
        code, outs = ops.request(place, api.Config(), gif_pages=frames, destructive=True, **kw)
        assert code == 0 and len(outs) == n
        outs = [a.copy() for a in outs]                                                # the layer's frames live until its next request
        host_in = [c.copy() for c in canvases]                                         # untouched frames are returned as views of these
        code2, want = ops.request(host_in, api.Config(), **kw)
        assert code2 == 0
        for k in range(n):
            ref_k = want[k] if want is not None and len(want) == n else canvases[k]
            assert np.array_equal(outs[k], ref_k), (kw, k)
            rq = {a: b for a, b in kw.items()}
            c3, _, ref = _oracle(orc, canvases[k], rq, {})
            assert c3 == 0 and np.array_equal(outs[k], ref), (kw, k)


def test_gif_expand_and_pack_golden_from_reference(gpu, orc):
    """tests/golden/golden_io_v1.npz — outputs of the reference's own advancedio.c (LoadGIF, IplToFI24/32, RunJob on GIF
    pages): sub-frames with the row[w] over-read, pages without a transparent colour (palette[-1]), every disposal."""
    io = G.load_io()
    for gif in io["gifs"]:
        frames = [G.fi_page(f) for f in gif["frames"]]
        for d in (0, 1):
            got = gpu.gif_expand(frames, gif["cw"], gif["ch"], bool(d))
            for k, (a, b) in enumerate(zip(got, gif["out"][d])):
                assert np.array_equal(a, b), (gif["cw"], gif["ch"], d, k)
    for pk in io["packs"]:
        for bits in (24, 32):
            code, _, out = _gpu_run(gpu, pk["img"], {}, dict(pack=bits))
            assert code == 0 and np.array_equal(out, pk[f"fi{bits}"])
    for job in io["jobs"]:
        gif = io["gifs"][job["gif"]]
        page = int([t for t in job["query"].split("&") if t.startswith("page")][0].split("=")[1])
        frames = [G.fi_page(f) for f in gif["frames"]]
        canvas = gpu.gif_expand(frames[:page + 1], gif["cw"], gif["ch"], True)[page]
        rq = G.split_query(job["query"])
        fmt = [t for t in job["query"].split("&") if t.startswith("format")][0].split("=")[1]
        rq["flatten"] = fmt in ("jpg", "ppm")                      # bridge.c:641-645
        rq["pack"] = {"tga": 32, "ppm": 24}.get(fmt, 0)            # bridge.c:680: FIF_BMP == 0 leaves through cvEncodeImage
        code, _, out = _gpu_run(gpu, canvas, {}, rq)
        assert code == 0 and np.array_equal(out, job["out"]), job["query"]


def test_strip_kernels_watermark_under_all_orientations(gpu, orc):
    """INTER_AREA (fractional and integer: the strip kernels) + each of the eight output orientations + a watermark at
    several gravities: the strip epilogue pulls the watermark rectangle back into the base frame to skip untouched rows
    and keeps an affine store line per column, both of which depend on the orientation."""
    wm = rnd_image(5, 9, 13, 4)
    orient = [[], ["flip=10"], ["flip=01"], ["flip=11"], ["rotate=90"], ["rotate=180"], ["rotate=270"], ["rotate=90", "flip=10"], ["flip=01", "rotate=270"]]
    for (h, w, c) in [(96, 160, 4), (90, 150, 3)]:
        img = smooth_image(h + c, h, w, c)
        for resize in ("50,31", "53,30", None):                    # fractional, integer 3x3 (150x90 -> 50x30 only for the 3-ch frame), none
            for gx, gy, ox, oy in [("r", "b", 3, 2), ("l", "t", 0, 0), ("c", "c", -4, 5), ("r", "t", 40, 1)]:
                kw = dict(watermark=wm, wm_gravity_x=gx, wm_gravity_y=gy, wm_offset_x=ox, wm_offset_y=oy, wm_opacity=70)
                for fl in orient:
                    rq = dict(resize=resize, filters=fl) if resize else dict(filters=fl)
                    if resize == "53,30":
                        rq["resize"] = "50,30" if (w, h) == (150, 90) else "40,24"
                    code, _, out = _gpu_run(gpu, img, kw, rq)
                    c2, _, ref = _oracle(orc, img, rq, kw)
                    assert code == c2, (rq, kw, code, c2)
                    if code == 0:
                        _assert_same(out, ref, (rq, gx, gy, ox, oy), False)


ORIENT = [[], ["flip=10"], ["flip=01"], ["rotate=90"], ["rotate=180"], ["rotate=270"], ["rotate=90", "flip=10"], ["flip=01", "rotate=270"]]


@pytest.mark.parametrize("c", [1, 3, 4])
def test_tile_kernels_orientations_sizes_and_packing(gpu, orc, c):
    """The TMA tile kernels of round 2 — fused blur (dp4a/dp2a, tiled in destination space), cubic tile, and the strip
    kernel's NN / LINEAR / index-map modes — on odd sizes that leave partial tiles on either side, under every output
    orientation, with a watermark and the encoder-side packings (destination channel count != source's)."""
    wm = rnd_image(5, 9, 13, 4)
    kw = dict(allow_experiments=True, max_filters=8, max_w=0, max_h=0, watermark=wm, wm_gravity_x="r", wm_gravity_y="b", wm_offset_x=3, wm_offset_y=2, wm_opacity=70)
    gathers = [dict(filters=["blur=0.7"]), dict(filters=["blur=2.3"]), dict(filters=["blur=3.2"]), dict(filters=["blur=4.1"]),
               dict(resize="150,101,up"), dict(resize="97,140,up"), dict(resize="200,30,up"),
               dict(resize="150,101,up", simple=True), dict(resize="31,23", simple=True),
               dict(resize="150,101,up", interp=1), dict(resize="41,29", interp=1),
               dict(crop="61px,37px,5px,3px"), dict()]
    n = 0
    for (h, w) in [(45, 70), (67, 131), (97, 33)]:
        img = smooth_image(h + w + c, h, w, c)
        for gi, g in enumerate(gathers):
            if c == 1 and "filters" in g:
                continue                                   # a gray frame is promoted before the blur: covered by c == 3
            for oi, fl in enumerate(ORIENT):
                rq = dict(g); rq["filters"] = list(g.get("filters", [])) + fl
                if (gi + oi) % 3 == 0: rq["filters"] = rq["filters"] + ["vignette=0.7"]
                if (gi + oi) % 4 == 1: rq["pack"] = 32 if oi % 2 else 24
                if (gi + oi) % 5 == 2: rq["flatten"] = True
                code, _, out = _gpu_run(gpu, img, kw, rq)
                c2, _, ref = _oracle(orc, img, rq, kw)
                if "crop" in g and w < 66:
                    assert code == c2 == 50, (rq, code, c2)        # the 61 px window at x = 5 does not fit the 33 px frame
                    continue
                assert code == c2 == 0, (rq, code, c2)
                _assert_same(out, ref, ((h, w, c), rq), _vig(img.shape, kw, rq))
                n += 1
    assert n > 200


def test_many_lut_filters_fall_back_instead_of_failing(gpu, orc):
    """ADVICE r1: a pass whose op list + LUTs push a tile kernel's shared-memory request over the opt-in limit must take the
    direct kernel, not fail the launch (imgproc_max_filters_count raised far above the default)."""
    img = smooth_image(3, 432, 768, 4)
    kw = dict(max_filters=400, max_w=0, max_h=0)
    many = ["gradmap=306090,eecc00", "gamma=1.1"] * 20 + ["gamma=0.9"] * 7          # 47 ops, 40 LUTs
    for rq in (dict(resize="79,45", filters=many), dict(filters=["blur=2.3"] + many[:46])):
        code, _, out = _gpu_run(gpu, img, kw, rq)
        c2, _, ref = _oracle(orc, img, rq, kw)
        assert code == c2 == 0, (code, c2, gpu.last_error())
        _assert_same(out, ref, rq["filters"][:2], False)
    # 3840x2160x4 -> resize=395: a 100 KB source tile + 2 ring stages + 33 KB of LUTs is over the limit
    big = smooth_image(4, 2160, 3840, 4)
    rq = dict(resize="395", filters=["gradmap=306090,eecc00"] * 40)
    code, _, out = _gpu_run(gpu, big, kw, rq)
    assert code == 0, gpu.last_error()
    _assert_same(out, _oracle(orc, big, rq, kw)[2], "resize=395 + 40 gradmaps", False)


def test_reference_runjob_with_the_gpu_path_dropped_in(gpu, orc):
    """The drop-in claim, executed: the reference's OWN RunJob (bridge.c:302-724), decode and encode included, compiled
    with INTEGRATION.md's call-site edits and linked against libimp_gpu.so (oracle/make_gpu_bridge.py ->
    oracle/_ref/libimp_ref_gpu.so), against the unmodified CPU build of the same sources (libimp_ref.so): same code,
    same failing step, same bytes, for single frames and for multi-frame GIF containers."""
    if not (orc.RefGpu.available() and orc.Ref.available()):
        pytest.skip("prebuilt oracle/_ref libraries not present on this box")
    from test_oracle import QUERIES
    wm = rnd_image(7, 12, 20, 4)
    cfgs = [orc.OracleConfig(), orc.OracleConfig(allow_experiments=True, max_filters=8),
            orc.OracleConfig(allow_experiments=True, max_filters=8, watermark=wm, wm_gravity_x="r", wm_gravity_y="b", wm_offset_x=3, wm_offset_y=2, wm_opacity=60)]
    checked = 0
    for (h, w, c) in [(60, 80, 3), (45, 64, 4), (33, 47, 1)]:
        img = smooth_image(h, h, w, c)
        for cfg in cfgs:
            for q in QUERIES:
                pc, p = orc.parse_query(q, cfg)
                # the CPU reference double-frees a frame when a filter fails after gray->BGR / flip / rotate (bridge.c:609-627)
                if not pc:
                    c2, s2, _ = orc.run_chain(img, p["crop"], p["gravity"], p["resize"], p["filters"], cfg, False, flatten=(p["format"] == "jpg"))
                    if c2 and s2 == orc.STEP_FILTERING and (c == 1 or any(f and (f.startswith("flip") or f.startswith("rotate")) for f in p["filters"])):
                        continue
                code, step, ref = orc.Ref.run_job(q, img, cfg)
                gcode, gstep, out = orc.RefGpu.run_job(q, img, cfg)
                assert (gcode, gstep) == (code, step), (q, (h, w, c), gcode, gstep, code, step)
                if code == 0 and ref is not None:
                    _assert_same(out, ref, (q, (h, w, c)), _vig(img.shape, dict(vars(cfg)), G.split_query(q)))
                    checked += 1
    io = G.load_io()
    for gi, q in [(1, "page=5&resize=33,21&filter-modulate=0,0,100&filter-colorize=704214,0.6&format=png"), (4, "page=3&crop=16,9&gravity=r,b&resize=40&format=bmp"),
                  (0, "page=2&filter-flip=10&filter-gamma=0.8&format=ppm"), (1, "page=6&resize=200,150,up&format=jpg"), (3, "page=1&resize=9,9&format=tga"),
                  (2, "page=1&format=png"), (0, "resize=24,14&format=gif"), (4, "filter-rotate=90&format=gif")]:
        blob = orc.Ref.gif_container(io["gifs"][gi]["frames"])
        code, step, ref = orc.Ref.run_job_blob(q, blob)
        raw = orc.Ref.last_raw
        gcode, gstep, out = orc.RefGpu.run_job_blob(q, blob)
        assert (gcode, gstep) == (code, step) and code == 0, (q, gcode, gstep, code, step)
        if ref is not None:
            _assert_same(out, ref, q, False)
        else:                                   # format=gif: every frame, through SaveGIF's (stand-in) quantiser
            assert len(raw) > 12 and orc.RefGpu.last_raw == raw, q
        checked += 1
    # a GIF request that fails AFTER LoadGIF handed its pages over (the frames are released unflushed), then ordinary requests:
    # the stale page registry of the drop-in must not claim a later album whose frame happens to live at a recycled address
    blob = orc.Ref.gif_container(io["gifs"][1]["frames"])
    for bad in ("crop=0,0&format=gif", "resize=0,0&format=gif", "filter-nosuchfilter=1&format=gif"):
        code, step, _ = orc.Ref.run_job_blob(bad, blob)
        gcode, gstep, _ = orc.RefGpu.run_job_blob(bad, blob)
        assert (gcode, gstep) == (code, step) and code != 0, (bad, gcode, gstep, code, step)
        for (h, w, c) in [(60, 80, 4), (45, 64, 4), (33, 47, 3)]:
            img = smooth_image(h + 1, h, w, c)
            q = "resize=31,17&filter-gamma=1.2&format=png"
            code, step, ref = orc.Ref.run_job(q, img, cfgs[0])
            gcode, gstep, out = orc.RefGpu.run_job(q, img, cfgs[0])
            assert (gcode, gstep) == (code, step) and code == 0
            _assert_same(out, ref, (bad, q, (h, w, c)), False)
            checked += 1
    assert checked > 150


def test_long_filter_lists_split_into_passes(gpu, orc):
    """More ops than one pass holds (48) or more tables than its shared memory takes: the chain continues in an index-map
    pass (gather tile kernel over the L2-resident scratch) instead of failing with TOO_MUCH_FILTERS (ADVICE r1)."""
    img = smooth_image(4, 140, 256, 4)
    kw = dict(allow_experiments=True, max_filters=200, max_w=0, max_h=0)
    chains = [["modulate=10,90,100", "rainbow=pale"] * 30,
              ["gotham=1"] * 20 + ["rotate=90"] + ["kelvin=1"] * 15 + ["scanline=0.5,0.25,1,1"] * 20,
              ["blur=1"] + ["lomo=1", "gamma=1.1", "vignette=0.6"] * 25 + ["blur=0.5"],
              ["gradmap=306090,eecc00", "gamma=1.1"] * 45]
    for f in chains:
        for rq in (dict(resize="130,70", filters=f), dict(filters=f, flatten=True)):
            code, _, out = _gpu_run(gpu, img, kw, rq)
            c2, _, ref = _oracle(orc, img, rq, kw)
            assert code == c2 == 0, (code, c2, gpu.last_error())
            _assert_same(out, ref, f[:3], _vig(img.shape, kw, rq))
