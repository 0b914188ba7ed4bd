"""
Generates tests/golden/golden_cv2_v1.json: what OpenCV's own resize, Gaussian blur, flip, transpose and rotate return for
the inputs of tests/test_oracle.py's cv2 cases (tests/golden_util.py: cv2_resize_cases, cv2_gaussian_cases,
cv2_orient_image). cv2 4.13.0 with IPP off stands in for the OpenCV calls the reference makes (it pins 2.4.9; SURVEY §8c).
The results are stored as SHA-256 digests of shape and bytes (about 3.5 MB of frames in full), beside the digest of each input,
so a changed random stream shows up as an input mismatch rather than as a wrong result.
Run:  python tests/golden/make_golden_cv2.py        (needs cv2 4.13)
"""
import json
import os
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import golden_util as G  # noqa: E402


def main():
    assert cv2.__version__.startswith("4.13."), cv2.__version__
    cv2.ipp.setUseIPP(False)
    cv2.setNumThreads(1)
    cases = {}

    def put(key, img, out):
        cases[key] = {"in": G.digest(img), "out": G.digest(out)}

    for key, img, dw, dh, mode in G.cv2_resize_cases():
        put(key, img, cv2.resize(img, (dw, dh), interpolation=mode).reshape(dh, dw, img.shape[2]))
    for key, img, sigma in G.cv2_gaussian_cases():
        out = cv2.GaussianBlur(img, (0, 0), float(np.float32(sigma)), sigmaY=0, borderType=cv2.BORDER_REPLICATE)
        put(key, img, out.reshape(img.shape))
    img = G.cv2_orient_image()
    for m in (0, 1, -1):
        put(f"flip/{m}", img, cv2.flip(img, m))
    put("transpose", img, cv2.transpose(img))
    put("rotate90", img, cv2.rotate(img, cv2.ROTATE_90_CLOCKWISE))
    with open(G.CV2_PATH, "w") as f:
        json.dump({"cv2": cv2.__version__, "ipp": False, "cases": cases}, f, indent=0, sort_keys=True)
        f.write("\n")
    print(G.CV2_PATH, os.path.getsize(G.CV2_PATH), "bytes,", len(cases), "cases")


if __name__ == "__main__":
    main()
