"""CPU tests of the product's HOST logic: the planner (argument grammar, return codes, lowering into
passes, frame-map algebra, tables) and the exact per-pixel source the CUDA kernels compile, walked on the
CPU by tests/hostsim (test-only; not a fallback) and compared with the oracle and the golden vectors."""
import numpy as np
import pytest

import golden_util as G
from conftest import rnd_image, smooth_image
from ngx_http_imgproc_b200 import api


def _oracle(orc, img, rq, cfgkw):
    ocfg = orc.OracleConfig(**cfgkw)
    o = dict(rq)
    interp = o.pop("interp", 0)
    if len(o.get("filters", [])) > ocfg.max_filters:
        return 55, 0, None
    return orc.run_chain(img, o.get("crop"), o.get("gravity"), o.get("resize"), o.get("filters", []), ocfg,
                         o.get("simple", False), o.get("flatten", False), linear=bool(interp), pack=o.get("pack", 0))


@pytest.mark.parametrize("case", G.load(), ids=lambda c: c["name"])
def test_hostsim_matches_golden(hostsim, case):
    req = G.split_query(case["query"])
    code, step, out = hostsim.run(case["img"], api.Config(**case["cfgkw"]), **req)
    assert code == case["code"]
    if code:
        assert step == case["step"] or code == 55
        return
    assert out.shape == case["out"].shape
    if "vignette" in case["query"]:
        G.assert_vignette_exact(out, case["out"], case["img"].shape, case["cfgkw"], req, case["name"])
    else:
        assert np.array_equal(out, case["out"])


REQS = [dict(resize="30,20"), dict(crop="1,1"), dict(crop="16,9,l,t"), dict(crop="40px,20px,6px,0px"), dict(crop="40px,20"),
        dict(crop="5000px,10px"), dict(crop="0px,10px"), dict(crop="10px,10px,x,t"), dict(crop="10px,10px,70px,0px"),
        dict(crop="1,1", gravity="r"), dict(crop="1,1", gravity="r,b"), dict(crop="3,2", gravity="c,c"), dict(crop="2,3,r,b"),
        dict(crop="10px,10px,-3px,0px"), dict(crop="1,1", gravity=",,,"),
        dict(resize="0,0"), dict(resize=""), dict(resize="100"), dict(resize="100,60"), dict(resize="0,30"), dict(resize="140,0,up"),
        dict(resize="3000,0,up"), dict(resize="120,90,up"), dict(crop="60px,40px,c,c", resize="20,10", filters=["gamma=1.3"]),
        dict(resize="33,21", filters=["modulate=0,0,100", "colorize=704214,0.6"]), dict(filters=["blur=2.3", "vignette=0.8", "rotate=90"]),
        dict(filters=["a=1", "b=1", "c=1", "d=1", "e=1", "f=1"]), dict(filters=["scanline=0.5,0.25,1,1", "flip=10", "rotate=270", "contrast=1.2"]),
        dict(filters=["flip=10", "gamma=0.8", "rotate=270", "contrast=1.2"]), dict(resize="200,150,up", filters=["lomo=1"]),
        dict(crop="1,1", resize="16", flatten=True), dict(resize="50", flatten=True, filters=["gotham=1"]), dict(filters=["gamma"]),
        dict(filters=["gamma="]), dict(resize="24,30", simple=True), dict(resize="90,70,up", simple=True),
        dict(filters=["rotate=90", "vignette=0.7", "flip=01", "scanline=0.4,0.3,2,1", "rotate=180", "blur=1.1", "rotate=270", "kelvin=1"]),
        dict(resize="40,30", filters=["blur=0.8", "rainbow=mid", "blur=1.5", "gradmap=306090,eecc00"]),
        dict(resize="31,17", filters=["rotate=270", "vignette=0.9,0.8"]), dict(resize="40,20"), dict(resize="20,15"), dict(resize="40,60"),
        dict(resize="16,12", interp=1), dict(resize="100,77,up", interp=1), dict(resize="32,24", interp=1),
        dict(filters=["blur=0"]), dict(filters=["scanline=,"]), dict(filters=["gradmap=306090"]), dict(filters=["vignette=,"]),
        dict(filters=["contrast=1e30"]), dict(filters=["modulate=0,-50,100"]), dict(filters=["modulate=77,0,250"]), dict(filters=["modulate=10,0,-30"]),
        dict(filters=["modulate=180,0,0"]), dict(filters=["modulate=0,0,99", "modulate=5,100,100"]), dict(filters=["gamma=0"]), dict(filters=["gamma=-1"]),
        # encoder-side packing (advancedio.c:65-101): bottom-up 24/32-bit
        dict(resize="40,30", pack=24), dict(resize="40,30", pack=32), dict(filters=["rotate=90", "blur=1.2"], pack=32),
        dict(crop="1,1", filters=["flip=10"], pack=24, flatten=True)]


def test_hostsim_matches_oracle_matrix(hostsim, orc):
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
                code, step, out = hostsim.run(img, api.Config(**kw), **rq)
                c2, s2, o2 = _oracle(orc, img, rq, kw)
                assert code == c2, (ci, rq)
                if code:
                    assert step == s2, (ci, rq)
                else:
                    assert out.shape == o2.shape and np.array_equal(out, o2), (ci, (h, w, c), rq)
                n += 1
    assert n > 800


def test_watermark_off_image_is_invalid_args(hostsim, orc):
    img = rnd_image(1, 20, 30, 3)
    kw = dict(watermark=rnd_image(2, 5, 5, 4), wm_gravity_x="l", wm_gravity_y="t", wm_offset_x=40, wm_offset_y=0)
    assert hostsim.run(img, api.Config(**kw))[:2] == (50, 6)
    assert _oracle(orc, img, {}, kw)[:2] == (50, 6)


def test_long_filter_lists_split_into_passes_and_validate_mode_agrees(hostsim, orc):
    """ADVICE r1: the reference takes as many filters as imgproc_max_filters_count allows; a pass holds 48 ops, so a longer
    chain continues in an index-map pass instead of failing with 55. Channel-separable runs (gotham's colorize + gamma +
    contrast, a sepia's modulate(s=0) + colorize) are one fused table op each. The validate-only mode of the planner (what
    every recorded operator of the imp_ops layer runs) returns the same code and geometry as the full lowering."""
    import ctypes as C
    img = smooth_image(4, 40, 56, 4)
    kw = dict(allow_experiments=True, max_filters=200, max_w=0, max_h=0)
    chains = [["modulate=10,90,100", "rainbow=pale"] * 30,                              # 60 ops that cannot fuse: two passes
              ["gotham=1"] * 20 + ["rotate=90"] + ["kelvin=1"] * 15 + ["scanline=0.5,0.25,1,1"] * 20,
              ["blur=1"] + ["lomo=1", "gamma=1.1", "vignette=0.6"] * 25 + ["blur=0.5"],
              ["gradmap=306090,eecc00", "gamma=1.1"] * 45]                              # 45 tables: the table area splits it too
    for f in chains:
        rq = dict(resize="30,20", filters=f)
        code, step, out, info = hostsim.run(img, api.Config(**kw), want_info=True, **rq)
        c2, s2, ref = _oracle(orc, img, rq, kw)
        assert code == c2 == 0
        G.assert_vignette_exact(out, ref, img.shape, kw, rq, f[:3])
    assert hostsim.run(img, api.Config(**kw), want_info=True, filters=chains[0])[3]["passes"] == 2
    one = hostsim.run(img, api.Config(**kw), want_info=True, filters=["gotham=1", "modulate=0,0,100", "colorize=704214,0.6", "contrast=1.2"])[3]
    assert one["passes"] == 1
    # validate-only mode == full mode on the whole request matrix's codes and geometry
    hostsim.lib.hostsim_plan_validate.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    n = 0
    for rq in REQS + [dict(filters=c) for c in chains]:
        for shape in [(60, 80, 3), (33, 47, 1), (45, 64, 4)]:
            cfg = api.Config(**(kw if "filters" in rq and len(rq["filters"]) > 8 else dict(allow_experiments=True, max_filters=8)))
            ccfg, k1 = cfg.to_c(); creq, k2 = api.make_request(**rq)
            step, out3 = C.c_int(-1), (C.c_int * 3)()
            rc = hostsim.lib.hostsim_plan_validate(C.byref(creq), C.byref(ccfg), shape[1], shape[0], shape[2], C.byref(step), out3)
            full = hostsim.run(np.zeros(shape, np.uint8), cfg, **rq)
            assert rc == full[0] and (rc == 0 or step.value == full[1]), (rq, shape, rc, full[:2])
            if rc == 0:
                assert tuple(out3) == (full[2].shape[1], full[2].shape[0], full[2].shape[2]), (rq, shape)
            n += 1
    assert n > 90


def test_plan_structure_and_algorithmic_bytes(hostsim):
    """One pass unless a blur splits the chain; SURVEY §8d byte counts for the five BASELINE configs."""
    img = np.zeros((108, 192, 3), np.uint8)
    _, _, _, info = hostsim.run(img, want_info=True, resize="64,36")
    assert info["passes"] == 1 and info["kinds"] == [2]                 # AREA_INT 3x3
    assert info["bytes"] == 192 * 108 * 3 + 64 * 36 * 3
    img4 = np.zeros((216, 384, 4), np.uint8)
    wm = np.zeros((8, 16, 4), np.uint8)
    _, _, _, info = hostsim.run(img4, api.Config(watermark=wm, wm_gravity_x="r", wm_gravity_y="b", wm_offset_x=1, wm_offset_y=1, wm_opacity=60),
                                want_info=True, crop="360px,202px,c,c", resize="80,45")
    assert info["passes"] == 1 and info["kinds"] == [3]                 # AREA_FRAC
    assert info["bytes"] == 360 * 202 * 4 + 80 * 45 * 4 + 16 * 8 * 4
    _, _, out, info = hostsim.run(np.zeros((40, 30, 3), np.uint8), api.Config(allow_experiments=True), want_info=True,
                                  filters=["blur=2.3", "vignette=0.8", "rotate=90"])
    assert info["passes"] == 1 and info["kinds"] == [6] and out.shape == (30, 40, 3)   # blur reads the source directly
    _, _, _, info = hostsim.run(np.zeros((40, 30, 3), np.uint8), want_info=True, resize="20,20", filters=["gamma=2", "blur=1", "blur=2"])
    assert info["passes"] == 3 and info["kinds"] == [3, 6, 6]
    _, _, out, info = hostsim.run(np.zeros((27, 48, 4), np.uint8), want_info=True, resize="96,54,up", filters=["modulate=0,0,100", "colorize=704214,0.6"])
    assert info["kinds"] == [4] and out.shape == (54, 96, 4)


def test_error_code_matrix_appendix_e(hostsim):
    """SURVEY Appendix E, through the product's planner."""
    img = rnd_image(3, 40, 60, 3)
    on, off = api.Config(allow_experiments=True), api.Config()
    def code(cfg=off, **rq): return hostsim.run(img, cfg, **rq)[0]
    for f in ["flip=00", "flip=01", "flip=10", "flip=11", "rotate=90", "rotate=180", "rotate=270", "modulate=0,-50,100", "colorize=ff0000,0", "gamma=0"]:
        assert code(filters=[f]) == 0, f
    for f in ["flip=2", "flip=12", "rotate=45", "modulate=181,1,1", "modulate=1,1,0", "modulate=1,1", "colorize=fff", "colorize=ff0000,1.5",
              "blur=-1", "contrast=0", "contrast=-1", "gradmap=12345", "gamma", "gamma="]:
        assert code(filters=[f]) == 50, f
    for f in ["rainbow=foo", "scanline=2", "scanline=0.5,2", "scanline=0.5,0,0"]:
        assert code(on, filters=[f]) == 50, f
    for f in ["vignette=0.8", "gotham=1"]:
        assert code(filters=[f]) == 52 and code(on, filters=[f]) == 0
    for f in ["nope=1", "cartoon=1", "Gamma=1"]:
        assert code(on, filters=[f]) == 52
    assert code(filters=["gamma=1"] * 6) == 55
    for c in ["1,1", "16,9,l,t", "40px,20px,6px,0px"]:
        assert code(crop=c) == 0
    for c in ["40px,20", "5000px,10px", "0px,10px", "10px,10px,x,t", "10px,10px,55px,0px"]:
        assert code(crop=c) == 50
    # pixel offsets near INT_MAX must not wrap past the window check (ADVICE r1: they reached the kernels as win_x = 2^31-1)
    for c in ["10px,10px,2147483647px,0px", "10px,10px,0px,2147483647px", "10px,10px,4294967295px,0px", "10px,10px,2147483640px,2147483640px"]:
        assert code(crop=c) == 50, c
    assert code(crop="10px,10px", gravity="2147483647px,0px") == 50 and code(crop="10px,10px", gravity="0px,2147483647px") == 50
    assert code(crop="1,1", gravity="r") == 50 and code(crop="1,1", gravity="r,b") == 0
    assert code(resize="0,0") == 50 and code(resize="") == 50
    for r in ["100", "100,60", "0,30", "140,0,up"]:
        assert code(resize=r) == 0
    assert code(resize="3000,0,up") == 54


def test_hostsim_random_requests_vs_oracle(hostsim, orc):
    """Random requests (crop, every resize flavour, up to four filters, watermark, flatten, FI packing) through the planner
    and the kernels' own per-pixel headers walked on the CPU, against the oracle: the CPU-box twin of scratch/fuzz_gpu.py."""
    rng = np.random.default_rng(2024)
    filt = ["flip=10", "flip=01", "rotate=90", "rotate=180", "rotate=270", "modulate=30,120,90", "modulate=12,0,140", "colorize=336699,0.4", "gamma=0.7",
            "contrast=1.3", "gradmap=102030,f0e0d0", "vignette=0.7", "gotham=1", "lomo=1", "kelvin=1", "rainbow=mid", "scanline=0.6,0.2,2,1",
            "blur=0.6", "blur=1.4", "blur=2.3"]
    done = 0
    for it in range(160):
        c = int(rng.choice([1, 3, 4])); h = int(rng.integers(1, 70)); w = int(rng.integers(1, 90))
        img = rng.integers(0, 256, (h, w, c), dtype=np.uint8)
        rq = {}
        if rng.random() < 0.4:
            cw, ch = int(rng.integers(1, w + 1)), int(rng.integers(1, h + 1))
            rq["crop"] = f"{cw}px,{ch}px,{int(rng.integers(0, w - cw + 1))}px,{int(rng.integers(0, h - ch + 1))}px"
        if rng.random() < 0.7:
            rq["resize"] = f"{int(rng.integers(1, 120))},{int(rng.integers(1, 100))}" + (",up" if rng.random() < 0.5 else "")
            if rng.random() < 0.15: rq["simple"] = True
            if rng.random() < 0.15: rq["interp"] = 1
        rq["filters"] = [str(f) for f in rng.choice(filt, int(rng.integers(0, 5)))]
        if rng.random() < 0.3: rq["flatten"] = True
        if rng.random() < 0.2: rq["pack"] = int(rng.choice([24, 32]))
        kw = dict(allow_experiments=True, max_filters=8, max_w=0, max_h=0)
        if rng.random() < 0.4:
            kw.update(watermark=rng.integers(0, 256, (int(rng.integers(1, 20)), int(rng.integers(1, 25)), int(rng.choice([3, 4]))), dtype=np.uint8),
                      wm_gravity_x=str(rng.choice(list("lcr"))), wm_gravity_y=str(rng.choice(list("tcb"))),
                      wm_offset_x=int(rng.integers(-8, 12)), wm_offset_y=int(rng.integers(-8, 12)), wm_opacity=int(rng.integers(1, 101)))
        code, step, out = hostsim.run(img, api.Config(**kw), **rq)
        c2, s2, o2 = _oracle(orc, img, rq, kw)
        assert code == c2, (it, rq, code, c2)
        if code:
            assert step == s2, (it, rq)
            continue
        if any("vignette" in f for f in rq["filters"]):
            G.assert_vignette_exact(out, o2, img.shape, kw, rq, (it, (h, w, c), rq))
        else:
            assert np.array_equal(out, o2), (it, (h, w, c), rq)
        done += 1
    assert done > 100
