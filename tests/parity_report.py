"""Parity report (GPU box): max |diff| and PSNR of the CUDA path against the CPU oracle for the five BASELINE configs
and every filter, through the C ABI. Test infrastructure: `python tests/parity_report.py > profiles/r01_parity_report.txt`.
PSNR is reported as 'inf' for bit-exact results. The test-suite enforces 0 everywhere; a vignette may differ by 1 only at pixels whose mask rounding is ambiguous (tests/vignette_ref.py)."""
import math
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE)); sys.path.insert(0, HERE)
import ngx_http_imgproc_b200 as M                    # noqa: E402
from ngx_http_imgproc_b200 import api                # noqa: E402
from oracle import oracle as O                       # noqa: E402
from conftest import rnd_image, smooth_image         # noqa: E402
from test_planner_host import _oracle                # noqa: E402
from test_gpu_parity import _gpu_run, FILTERS        # noqa: E402


def psnr(a, b):
    mse = float(np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2))
    return "inf" if mse == 0 else "%.2f" % (10 * math.log10(255.0 ** 2 / mse))


def line(name, out, ref):
    d = np.abs(out.astype(int) - ref.astype(int))
    print(f"{name:78s} {out.shape[1]:5d}x{out.shape[0]:<5d}x{out.shape[2]}  max|d|={int(d.max())}  differing={int((d > 0).sum())}/{d.size}  PSNR={psnr(out, ref)} dB")


def main():
    L = M.library(); L.init(0)
    wm = rnd_image(3, 64, 256, 4); wm[:, :, 3] = np.linspace(0, 255, 256).astype(np.uint8)[None, :]
    wkw = dict(watermark=wm, wm_gravity_x="r", wm_gravity_y="b", wm_offset_x=10, wm_offset_y=10, wm_opacity=60)
    cases = [
        ("cfg1 1080p -> 640x360 INTER_AREA (the reference's call)", rnd_image(1, 1080, 1920, 3), {}, dict(resize="640,360")),
        ("cfg1 1080p -> 640x360 INTER_LINEAR (extension)", rnd_image(1, 1080, 1920, 3), {}, dict(resize="640,360", interp=1)),
        ("cfg2 4K BGRA crop 3600x2025 -> AREA 800x450 + watermark", smooth_image(2, 2160, 3840, 4), wkw, dict(crop="3600px,2025px,c,c", resize="800,450")),
        ("cfg3 480x270 BGRA -> cubic 2x + sepia", smooth_image(4, 270, 480, 4), {}, dict(resize="960,540,up", filters=["modulate=0,0,100", "colorize=704214,0.6"])),
        ("cfg3 480x270 BGRA -> NN 2x + sepia (GIF output path)", smooth_image(4, 270, 480, 4), {}, dict(resize="960,540,up", simple=True, filters=["modulate=0,0,100", "colorize=704214,0.6"])),
        ("cfg4 12 MP blur=2.3 + vignette=0.8 + rotate=90", smooth_image(5, 3000, 4000, 3), dict(allow_experiments=True), dict(filters=["blur=2.3", "vignette=0.8", "rotate=90"])),
        ("cfg5 1600x1200 -> 256x256 AREA + 64x64 watermark", rnd_image(6, 1200, 1600, 3),
         dict(max_w=0, max_h=0, watermark=rnd_image(61, 64, 64, 4), wm_gravity_x="r", wm_gravity_y="b", wm_offset_x=8, wm_offset_y=8, wm_opacity=100), dict(resize="256,256")),
    ]
    for name, img, kw, rq in cases:
        code, _, out = _gpu_run(L, img, kw, rq)
        c2, _, ref = _oracle(O, img, rq, kw)
        assert code == c2 == 0, (name, code, c2)
        line(name, out, ref)
    img = rnd_image(77, 240, 320, 4)
    for f in FILTERS:
        kw = dict(allow_experiments=True, max_filters=8)
        code, _, out = _gpu_run(L, img, kw, dict(filters=[f]))
        c2, _, ref = _oracle(O, img, dict(filters=[f]), kw)
        assert code == c2 == 0, f
        line("filter " + f, out, ref)


if __name__ == "__main__":
    main()
