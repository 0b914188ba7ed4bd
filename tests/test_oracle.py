"""CPU tests of the oracle: the C restatement against (1) SURVEY App. B known answers, (2) the golden
vectors generated from the compiled reference + cv2 and the stored cv2 4.13 results (tests/golden/), (3) live,
the compiled reference (oracle/_ref, built from the reference's sources by oracle/Makefile) when it is present."""
import numpy as np
import pytest

import golden_util as G
from conftest import rnd_image, smooth_image

KAT = np.array([[[0, 0, 0], [255, 255, 255], [10, 128, 250], [200, 30, 180]],
                [[37, 201, 99], [128, 128, 128], [255, 0, 170], [3, 2, 1]]], np.uint8)

APP_B = {   # SURVEY Appendix B (compiled reference, gcc -O1)
    "modulate=0,0,100": [[0,0,0],[255,255,255],[250,250,250],[200,200,200],[201,201,201],[128,128,128],[255,255,255],[3,3,3]],
    "modulate=60,70,80": [[0,0,0],[204,204,204],[128,200,66],[65,147,160],[160,102,69],[102,102,102],[61,156,204],[1,1,2]],
    "modulate=100,500,500": [[0,0,0],[255,255,255],[255,51,0],[51,255,0],[255,0,246],[255,255,255],[0,255,0],[0,12,15]],
    "colorize=704214,0.6": [[12,39,67],[113,141,169],[16,90,167],[91,51,139],[26,120,106],[63,90,118],[113,39,135],[13,40,67]],
    "colorize=ff0000": [[0,0,127],[127,127,255],[5,64,252],[100,15,217],[18,100,177],[64,64,191],[127,0,212],[1,1,128]],
    "gamma=1.3": [[0,0,0],[255,255,255],[21,150,251],[211,49,195],[57,212,123],[150,150,150],[255,0,186],[8,6,3]],
    "gamma=0.5": [[0,0,0],[255,255,255],[0,64,245],[156,3,127],[5,158,38],[64,64,64],[255,0,113],[0,0,0]],
    "contrast=1.5": [[0,0,0],[255,255,255],[15,192,255],[255,45,255],[55,255,148],[192,192,192],[255,0,255],[4,3,1]],
    "contrast=0.5": [[0,0,0],[127,127,127],[5,64,125],[100,15,90],[18,100,49],[64,64,64],[127,0,85],[1,1,0]],
    "gradmap=306090,eecc00": [[144,96,48],[1,204,237],[71,150,144],[68,153,149],[81,143,131],[72,150,143],[65,155,153],[143,97,49]],
    "vignette=0.8": [[0,0,0],[149,149,149],[8,94,192],[117,17,103],[11,65,31],[98,98,98],[255,0,169],[2,1,0]],
    "vignette=4,3": [[0,0,0],[49,49,49],[5,57,117],[39,5,34],[0,3,1],[59,59,59],[255,0,169],[1,0,0]],
    "gotham=1": [[0,0,0],[252,214,211],[237,169,178],[105,88,70],[100,76,85],[13,6,4],[241,214,178],[0,0,0]],
    "lomo=1": [[0,0,0],[255,255,255],[10,142,255],[200,0,220],[37,251,98],[128,142,142],[255,0,205],[3,0,0]],
    "kelvin=1": [[0,76,127],[127,204,255],[125,141,220],[94,176,185],[74,136,228],[64,140,191],[106,204,191],[0,78,128]],
    "rainbow=full": [[0,0,0],[255,255,255],[0,125,250],[200,0,146],[0,201,0],[0,0,128],[255,255,255],[0,0,0]],
    "rainbow=pale": [[0,0,0],[255,255,255],[132,191,250],[200,105,174],[106,201,106],[67,67,128],[255,255,255],[0,0,0]],
    "scanline=0.5,0.25,1,1": [[0,0,0],[255,255,255],[10,122,250],[200,30,177],[95,127,107],[95,95,127],[127,95,116],[127,111,95]],
}


@pytest.mark.parametrize("req", sorted(APP_B))
def test_appendix_b_known_answers(orc, req):
    code, out = orc.apply_filter(KAT, req, True)
    assert code == 0
    assert out.reshape(-1, 3).tolist() == APP_B[req]


def test_appendix_b_hsv_and_sepia(orc):
    o = orc.orc()
    assert o.rgb2hsv(KAT).reshape(-1, 3).tolist() == [[0,0,0],[0,0,255],[14,244,250],[146,216,200],[49,208,201],[0,0,128],[140,255,255],[105,170,3]]
    assert o.hsv2rgb(o.rgb2hsv(KAT)).reshape(-1, 3).tolist() == [[0,0,0],[255,255,255],[10,122,250],[200,30,177],[37,201,97],[128,128,128],[255,0,169],[3,1,0]]
    code, step, sep = orc.run_chain(KAT, filters=["modulate=0,0,100", "colorize=704214,0.6"])
    assert sep.reshape(-1, 3).tolist() == [[12,39,67],[113,141,169],[111,139,167],[91,119,147],[92,120,147],[63,90,118],[113,141,169],[13,40,68]]
    assert abs(o.perceived_brightness(KAT) - 0.45781034) < 1e-6


def test_appendix_b_compositing(orc):
    o = orc.orc()
    dst = np.array([[[10,20,30,255],[10,20,30,128],[10,20,30,0],[200,100,50,255]]], np.uint8)
    src = np.array([[[255,0,0,255],[0,255,0,128],[0,0,255,64],[90,90,90,0]]], np.uint8)
    assert o.alpha_over(dst, 0, 0, src, 1.0)[0].tolist() == [[255,0,0,255],[3,176,9,191],[0,0,254,64],[200,100,50,255]]
    assert o.alpha_over(dst, 0, 0, src, float(np.float32(0.6)))[0].tolist() == [[157,7,11,255],[8,63,24,140],[0,0,0,0],[200,100,50,255]]
    d3 = np.array([[[10,20,30],[200,100,50],[0,0,0],[255,255,255]]], np.uint8)
    assert o.alpha_over(d3, 0, 0, src, float(np.float32(0.6)))[0].tolist() == [[157,7,11],[179,115,44],[0,0,0],[255,255,255]]
    pp = np.array([[[10,20,30,255],[10,20,30,128],[10,20,30,0],[200,100,50,77]]], np.uint8)
    assert o.paper(pp)[0].tolist() == [[10,20,30,255],[132,137,142,255],[255,255,255,255],[238,208,193,255]]


def test_gaussian_taps_known_answers(orc):
    o = orc.orc()
    assert o.gaussian_taps(0.5) == [0, 27, 202, 27, 0]
    assert o.gaussian_taps(1.0) == [1, 14, 62, 102, 62, 14, 1]
    assert o.gaussian_taps(2.0) == [1, 2, 7, 16, 31, 45, 52, 45, 31, 16, 7, 2, 1]
    assert o.gaussian_taps(float(np.float32(2.3))) == [0, 2, 4, 10, 19, 30, 41, 44, 41, 30, 19, 10, 4, 2, 0]


def test_cubic_2x_phase_coefficients(orc):
    """App. A.4: exact 2x upscale has two phases (f = 0.75 / 0.25). With OpenCV's A = -0.75 the 11-bit sets are
    (-72,536,1800,-216)/(-216,1800,536,-72) (SURVEY's printed numbers correspond to A = -0.5; cv2 parity in
    test_restatement_vs_cv2_resize_fuzz pins A = -0.75)."""
    import ctypes as C
    L = orc.orc().lib
    ofs = (C.c_int * 8)(); coef = (C.c_short * 32)()
    L.orc_interp_tab.argtypes = [C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.orc_interp_tab(4, 8, 0.5, 1, 1, ofs, coef)
    assert list(coef[4:8]) == [-216, 1800, 536, -72] and list(coef[8:12]) == [-72, 536, 1800, -216]


@pytest.mark.parametrize("case", G.load(), ids=lambda c: c["name"])
def test_restatement_matches_golden(orc, case):
    """The restatement reproduces every golden vector (reference code, reference stage order, reference codes)."""
    cfg = orc.OracleConfig(**case["cfgkw"])
    pc, p = orc.parse_query(case["query"], cfg)
    if pc:
        assert pc == case["code"]
        return
    code, step, out = orc.run_chain(case["img"], p["crop"], p["gravity"], p["resize"], p["filters"], cfg, False, flatten=(p["format"] == "jpg"))
    assert code == case["code"]
    if code:
        assert step == case["step"]
    else:
        assert out.shape == case["out"].shape
        assert np.array_equal(out, case["out"])


# ---- live checks against the real things, when present (this container) ---------------------------------
def _have_ref(orc):
    return orc.Ref.available()


def _have_cv2():
    try:
        import cv2  # noqa: F401
        return True
    except Exception:
        return False


FILTER_REQS = ["flip=10", "flip=01", "flip=11", "flip=00", "rotate=90", "rotate=180", "rotate=270", "modulate=0,0,100", "modulate=60,70,80",
               "modulate=100,500,500", "modulate=180,-50,100", "modulate=1,1,1", "colorize=704214,0.6", "colorize=ff0000", "colorize=00ff7f,0",
               "colorize=123456,1", "blur=2.3", "blur=0.5", "blur=1", "gamma=1.3", "gamma=0.5", "gamma=2.2", "contrast=1.5", "contrast=0.5",
               "contrast=3.7", "gradmap=306090,eecc00", "gradmap=000000,ff0000,ffffff", "vignette=0.8", "vignette=4,3", "vignette=0.5,0.7",
               "gotham=1", "lomo=1", "kelvin=1", "rainbow=full", "rainbow=mid", "rainbow=pale", "scanline=0", "scanline=0.5,0.25,1,1",
               "scanline=0.3,0.9,2,3", "scanline=1,1,5,1",
               # Appendix E error matrix
               "flip=2", "flip=12", "rotate=45", "modulate=181,1,1", "modulate=1,1,0", "modulate=1,1", "colorize=fff", "colorize=ff0000,1.5",
               "blur=-1", "contrast=0", "contrast=-1", "gradmap=12345", "rainbow=foo", "scanline=2", "scanline=0.5,2", "scanline=0.5,0,0",
               "nope=1", "cartoon=1", "Gamma=1", "gamma", "gamma="]


@pytest.mark.parametrize("c", [3, 4])
def test_restatement_vs_compiled_reference_filters(orc, c):
    if not _have_ref(orc):
        pytest.skip("compiled reference not available on this box")
    for (h, w) in [(37, 53), (64, 64), (5, 3)]:
        img = rnd_image(h * w + c, h, w, c)
        for rq in FILTER_REQS:
            c1, a = orc.Ref.filter(img, rq, True)
            c2, b = orc.apply_filter(img, rq, True)
            assert c1 == c2, rq
            assert a.shape == b.shape and np.array_equal(a, b), rq
    for rq in ["vignette=0.8", "gotham=1", "lomo=1", "kelvin=1", "rainbow=full", "scanline=0.5"]:
        assert orc.Ref.filter(img, rq, False)[0] == orc.apply_filter(img, rq, False)[0] == 52


def _same_as_cv2(want, key, img, got):
    """got equals what cv2 4.13 returned for this input (tests/golden/golden_cv2_v1.json)."""
    assert G.digest(img) == want[key]["in"], (key, "the seeded input is not the one the golden results were made from")
    assert G.digest(got) == want[key]["out"], (key, img.shape, got.shape, "differs from cv2 4.13: compare pixel by pixel with cv2 "
                                               "on the same case (tests/golden/make_golden_cv2.py) to see where")


def test_restatement_vs_cv2_resize_fuzz(orc):
    want = G.load_cv2()
    o = orc.orc()
    keys = set()
    for key, img, dw, dh, mode in G.cv2_resize_cases():
        _same_as_cv2(want, key, img, o.resize(img, dw, dh, mode))
        keys.add(key)
    assert keys == {k for k in want if k.startswith("resize/")}


def test_restatement_vs_cv2_gaussian_and_index_maps(orc):
    want = G.load_cv2()
    o = orc.orc()
    keys = set()
    for key, img, sigma in G.cv2_gaussian_cases():
        _same_as_cv2(want, key, img, o.gaussian(img, sigma))
        keys.add(key)
    assert keys == {k for k in want if k.startswith("gaussian/")}
    img = G.cv2_orient_image()
    for m in (0, 1, -1):
        _same_as_cv2(want, f"flip/{m}", img, o.flip(img, m))
    _same_as_cv2(want, "transpose", img, o.transpose(img))
    _same_as_cv2(want, "rotate90", img, o.flip(o.transpose(img), 1))


QUERIES = ["resize=30,20", "crop=1,1", "crop=16,9,l,t", "crop=40px,20px,6px,0px", "crop=40px,20", "crop=5000px,10px", "crop=0px,10px",
           "crop=10px,10px,x,t", "crop=10px,10px,70px,0px", "crop=1,1&gravity=r", "crop=1,1&gravity=r,b", "crop=3,2&gravity=c,c",
           "crop=2,3,r,b", "resize=0,0", "resize=", "resize=100", "resize=100,60", "resize=0,30", "resize=140,0,up", "resize=3000,0,up",
           "resize=120,90,up", "crop=60px,40px,c,c&resize=20,10&filter-gamma=1.3",
           "resize=33,21&filter-modulate=0,0,100&filter-colorize=704214,0.6", "filter-blur=2.3&filter-vignette=0.8&filter-rotate=90",
           "filter-a=1&filter-b=1&filter-c=1&filter-d=1&filter-e=1&filter-f=1", "filter-scanline=0.5,0.25,1,1&filter-flip=10",
           "filter-flip=10&filter-gamma=0.8&filter-rotate=270&filter-contrast=1.2", "resize=200,150,up&filter-lomo=1",
           "crop=1,1&resize=16&format=jpg", "resize=50&format=jpg&filter-gotham=1", "filter-gamma", "filter-gamma=", "foo=bar"]


def test_restatement_vs_reference_runjob(orc):
    """Whole RunJob (bridge.c:302-724, RAW codec): same code, same failing step, same pixels."""
    if not _have_ref(orc):
        pytest.skip("compiled reference not available on this box")
    wm, wm3 = rnd_image(7, 12, 20, 4), rnd_image(8, 7, 9, 3)
    cfgs = [orc.OracleConfig(),
            orc.OracleConfig(allow_experiments=True, max_filters=8, watermark=wm, wm_gravity_x="r", wm_gravity_y="b", wm_offset_x=3, wm_offset_y=2, wm_opacity=60),
            orc.OracleConfig(allow_experiments=True, watermark=wm3, wm_gravity_x="c", wm_gravity_y="c", wm_offset_x=-4, wm_offset_y=5, wm_opacity=100),
            orc.OracleConfig(max_w=100, max_h=50, watermark=wm, wm_gravity_x="l", wm_gravity_y="t", wm_offset_x=-5, wm_offset_y=-3, wm_opacity=37)]
    for ci, cfg in enumerate(cfgs):
        for (h, w, c) in [(60, 80, 3), (45, 64, 4), (33, 47, 1)]:
            img = rnd_image(ci * 10 + c, h, w, c)
            for q in QUERIES:
                pc, p = orc.parse_query(q, cfg)
                if pc:
                    c2, s2, o2 = pc, 0, None
                else:
                    c2, s2, o2 = orc.run_chain(img, p["crop"], p["gravity"], p["resize"], p["filters"], cfg, False, flatten=(p["format"] == "jpg"))
                # The reference double-frees a frame when a filter fails after the image was replaced
                # (gray->BGR or flip/rotate): bridge.c:609-627 updates album.Frames[] only after the loop.
                if c2 and s2 == orc.STEP_FILTERING and (c == 1 or any(f and (f.startswith("flip") or f.startswith("rotate")) for f in p["filters"])):
                    continue
                code, step, out = orc.Ref.run_job(q, img, cfg)
                assert code == c2, (ci, q)
                if code:
                    assert pc or step == s2, (ci, q)
                else:
                    assert out.shape == o2.shape and np.array_equal(out, o2), (ci, q, (h, w, c))


def test_alpha_unit_identity():
    """(float)(a/255.0) == a/255.0f for every byte: the device uses one IEEE float division (imp_pixel.cuh)."""
    a = np.arange(256)
    assert np.array_equal((a / 255.0).astype(np.float32), a.astype(np.float32) / np.float32(255.0))


def test_ascii_restatement_vs_compiled_reference(orc):
    """SURVEY 8f-4: the restated ASCII equals the reference's (both ramps)."""
    if not _have_ref(orc):
        pytest.skip("compiled reference not available on this box")
    o = orc.orc()
    for (h, w, c) in [(7, 13, 3), (20, 31, 4), (1, 5, 3)]:
        img = rnd_image(h + w, h, w, c)
        for args, wide in (("wide", True), ("", False), ("narrow", False)):
            assert o.ascii(img, wide) == orc.Ref.ascii(img, args), (h, w, c, args)
    ramp = np.arange(256, dtype=np.uint8).reshape(1, 256, 1).repeat(3, 2)
    assert o.ascii(ramp, True) == orc.Ref.ascii(ramp, "wide") and o.ascii(ramp, False) == orc.Ref.ascii(ramp, "x")


# ---- advancedio.c: LoadGIF's canvas loop and IplToFI24/32, pinned against the reference's own code -------------------
def _gif_job_restated(orc, gif, query):
    """RunJob on a GIF with page=N, restated: destructive expansion up to the page, then steps 3-7, then the encoder's
    packing (cvEncodeImage RAW for png/jpg, IplToFI32 for bmp/tga, IplToFI24 for ppm)."""
    pc, p = orc.parse_query(query, orc.OracleConfig())
    assert pc == 0
    page = int([t for t in query.split("&") if t.startswith("page")][0].split("=")[1])
    frames = [G.fi_page(f) for f in gif["frames"]]
    canvas = orc.orc().gif_expand(frames[:page + 1], gif["cw"], gif["ch"], True)[page]
    # bridge.c:443-447,680: FIF_BMP == 0 reads as "no advanced encoder", so format=bmp leaves through cvEncodeImage;
    # bridge.c:641-645: formats without 32-bit support (ppm) are flattened like jpg.
    pack = {"tga": 32, "ppm": 24}.get(p["format"], 0)
    return orc.run_chain(canvas, p["crop"], p["gravity"], p["resize"], p["filters"], orc.OracleConfig(), False,
                         flatten=(p["format"] in ("jpg", "ppm")), pack=pack)


def test_gif_expand_and_pack_restatement_vs_golden(orc):
    """The committed vectors made from the reference's advancedio.c (tests/golden/make_golden_io.py)."""
    io = G.load_io()
    o = orc.orc()
    for gif in io["gifs"]:
        frames = [G.fi_page(f) for f in gif["frames"]]
        for d in (0, 1):
            got = o.gif_expand(frames, gif["cw"], gif["ch"], bool(d))
            for a, b in zip(got, gif["out"][d]):
                assert np.array_equal(a, b)
    for pk in io["packs"]:
        assert np.array_equal(orc.fi_pack(pk["img"], 24), pk["fi24"])
        assert np.array_equal(orc.fi_pack(pk["img"], 32), pk["fi32"])
    for job in io["jobs"]:
        code, _, out = _gif_job_restated(orc, io["gifs"][job["gif"]], job["query"])
        assert code == job["code"] == 0
        assert np.array_equal(out, job["out"]), job["query"]


def test_gif_expand_restatement_vs_reference_loadgif(orc):
    """Random multi-page GIFs through the reference's LoadGIF (advancedio.c compiled unmodified over the stand-in
    FreeImage): sub-frames, all disposal methods, pages with and without a transparent colour, destructive or not.
    The only pixel left out is the one the reference reads from beyond the page block (row[w] of the top scanline
    when w % 4 == 0), and whatever it feeds through `master` afterwards."""
    if not _have_ref(orc):
        pytest.skip("compiled reference not available on this box")
    rng = np.random.default_rng(1)
    o = orc.orc()
    compared = 0
    for trial in range(250):
        cw, ch, n = int(rng.integers(1, 24)), int(rng.integers(1, 20)), int(rng.integers(1, 6))
        fr = []
        for f in range(n):
            w, h = (cw, ch) if f == 0 else (int(rng.integers(1, cw + 1)), int(rng.integers(1, ch + 1)))
            left, top = (0, 0) if f == 0 else (int(rng.integers(0, cw - w + 1)), int(rng.integers(0, ch - h + 1)))
            dispose = int(rng.integers(0, 4))
            if f == 0 and dispose == 2:
                dispose = 1
            fr.append(dict(indices=rng.integers(0, 256 if rng.random() < .5 else 5, (h, w), dtype=np.uint8),
                           palette=rng.integers(0, 256, (256, 4), dtype=np.uint8), left=left, top=top, dispose=dispose,
                           key=int(rng.choice([-1, 0, 3, 255])), time=f))
        blob = orc.Ref.gif_container(fr)
        pages = [G.fi_page(f) for f in fr]
        for destructive in (False, True):
            err, ref = orc.Ref.fi_load(blob, orc.Ref.FIF_GIF, destructive)
            assert err == 0 and len(ref) == n
            got = o.gif_expand(pages, cw, ch, destructive)
            mask = np.ones((ch, cw), bool)
            for k in range(n):
                h, w = fr[k]["indices"].shape
                if not destructive:
                    mask[:] = True
                if w % 4 == 0 and fr[k]["left"] + w < cw:
                    mask[fr[k]["top"], fr[k]["left"] + w] = False
                assert not ((got[k] != ref[k]["image"]).any(axis=2) & mask).any(), (trial, destructive, k)
                assert (ref[k]["dispose"], ref[k]["key"]) == (fr[k]["dispose"], fr[k]["key"])
                compared += int(mask.sum())
    assert compared > 100000


def test_fi_pack_restatement_vs_reference_ipltofi(orc):
    """IplToFI32 / IplToFI24 (advancedio.c:65-101) through FiSaveFrames -> SaveSingle, 3- and 4-channel frames."""
    if not _have_ref(orc):
        pytest.skip("compiled reference not available on this box")
    for seed, (h, w, c) in enumerate([(5, 7, 3), (5, 7, 4), (1, 1, 3), (33, 18, 4), (16, 32, 3), (9, 13, 4)]):
        img = rnd_image(seed, h, w, c)
        for fmt, bits in ((orc.Ref.FIF_BMP, 32), (orc.Ref.FIF_TARGA, 32), (orc.Ref.FIF_JPEG, 24)):
            err, bpp, ref = orc.Ref.fi_save(img, fmt)
            assert err == 0 and bpp == bits
            assert np.array_equal(orc.fi_pack(img, bits), ref)


def test_runjob_on_gif_pages_vs_reference(orc):
    """Whole RunJob on GIF containers: the reference's FiLoadFrames + steps 3-7 + encoder against the restatement."""
    if not _have_ref(orc) or not _have_cv2():
        pytest.skip("needs the compiled reference and cv2")
    orc.Ref.use_cv2(True)
    io = G.load_io()
    try:
        for gi, q in [(1, "page=5&resize=33,21&filter-modulate=0,0,100&filter-colorize=704214,0.6&format=png"),
                      (4, "page=3&crop=16,9&gravity=r,b&resize=40&format=bmp"), (0, "page=2&filter-flip=10&filter-gamma=0.8&format=ppm"),
                      (1, "page=6&resize=200,150,up&format=jpg"), (3, "page=1&resize=9,9&format=tga"), (2, "page=1&format=png")]:
            gif = io["gifs"][gi]
            blob = orc.Ref.gif_container(gif["frames"])
            code, step, out = orc.Ref.run_job_blob(q, blob)
            c2, s2, o2 = _gif_job_restated(orc, gif, q)
            assert code == c2 == 0, (q, code, step)
            assert np.array_equal(out, o2), q
    finally:
        orc.Ref.use_cv2(False)


def test_integration_edits_apply_to_the_reference():
    """INTEGRATION.md's edits (oracle/make_gpu_bridge.py) still match the reference: the definitions imp_dropin.c replaces
    under their own names are cut out of bridge.c / filters.c, RunJob keeps every operator call site as the reference wrote
    it, loses the gray->BGR block and gains exactly one flush statement and one imp_Discard."""
    import importlib.util
    import os
    import re
    ref = "/root/reference/bridge.c"
    if not os.path.exists(ref):
        pytest.skip("reference sources not present on this box")
    here = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("make_gpu_bridge", os.path.join(here, "oracle", "make_gpu_bridge.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    src = open(ref).read()
    out = mod.patched_bridge(src)
    run_job = out[out.index("JobResult* RunJob"):]
    for kept in ("= Crop(&image, crop, gravity)", "= Resize(&image, resize, config, simple)", "= Filter(&image, filters[i], config->AllowExperiments)",
                 "= Watermark(image, config)", "\tBlendWithPaper(image);"):
        assert run_job.count(kept) == 1, kept                      # call sites untouched
    assert "CV_GRAY2BGR" not in run_job
    assert run_job.count("imp_FlushAlbum(&album)") == 1 and run_job.count("imp_Discard(image)") == 1
    for name in mod.BRIDGE_REPLACED:
        assert not re.search(r"^(?:int|void)\s+" + name + r"\s*\(", out, flags=re.M), name
    # what is left of the diff: the deleted bodies, one include + prototype, one block deleted, two statements
    removed = sum(1 for line in src.splitlines() if line.strip() and line not in out)
    assert removed > 150                                              # Crop + Resize + Watermark bodies are gone
    fsrc = open("/root/reference/filters.c").read()
    fout = mod.patched_filters(fsrc)
    for name in mod.FILTERS_REPLACED:
        assert not re.search(r"^(?:int|void)\s+" + name + r"\s*\(", fout, flags=re.M), name
    for kept in ("int Filter(", "int CheckDestructive(", "CallbackMap[]", "Memory ASCII", "float CalcPerceivedBrightness(", "void ModulateHSV("):
        assert kept in fout, kept
    # the shim defines exactly the symbols that were cut
    shim = open(os.path.join(here, "ngx_http_imgproc_b200", "dropin", "imp_dropin.c")).read()
    for name in mod.BRIDGE_REPLACED + mod.FILTERS_REPLACED:
        assert re.search(r"^(?:int|void)\s+" + name + r"\s*\(", shim, flags=re.M), name
    # INTEGRATION.md §4: LoadGIF loses its per-pixel canvas loop (and nothing else) to one imp_AlbumGifPage call
    asrc = open("/root/reference/advancedio.c").read()
    aout = mod.patched_advancedio(asrc)
    load_gif = aout[aout.index("static void LoadGIF("):aout.index("static void LoadSingle(")]
    assert load_gif.count("imp_AlbumGifPage(result, frameid, isdestructive,") == 1
    assert "cvSetComponent" not in load_gif and "master[offset]" not in load_gif
    for kept in ("FreeImage_LockPage(container, frameid)", "FreeImage_GetTransparentIndex(frame)", "FreeImage_ConvertTo8Bits(frame)",
                 "cvCreateImage(cvSize(canvasW, canvasH), IPL_DEPTH_8U, 4)", "FreeImage_UnlockPage(container, frame, 0)", "if (frameid == page)",
                 "result->Frames[0] = requested;"):
        assert kept in load_gif, kept
    gone = [l for l in asrc.splitlines() if l.strip() and l not in aout]
    assert 20 <= len(gone) <= 60, len(gone)                            # the loop nest only
    assert aout[aout.index("static void LoadSingle("):] == asrc[asrc.index("static void LoadSingle("):]
    assert re.search(r"^int\s+imp_AlbumGifPage\s*\(", shim, flags=re.M)
