"""Loads tests/golden/golden_v1.npz (made by tests/golden/make_golden.py from the compiled reference + cv2)."""
import hashlib
import json
import os
from urllib.parse import unquote

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_v1.npz")


def load():
    z = np.load(PATH)
    meta = json.loads(bytes(z["meta"]).decode())
    cases = []
    for i, m in enumerate(meta["cases"]):
        kw = {k: (z["WM"] if v == "WM" else v) for k, v in meta["cfg"][m["cfg"]].items()}
        cases.append(dict(m, img=z[f"in{i}"], out=(z[f"out{i}"] if f"out{i}" in z.files else None), cfgkw=kw))
    return cases


def split_query(query):
    """RunJob's query scan (bridge.c:346-372) for the keys the hot path uses. Returns request kwargs + format."""
    req = dict(crop=None, gravity=None, resize=None, filters=[])
    fmt = None
    for tok in [t for t in query.split("&") if t]:
        if tok.startswith("crop"): req["crop"] = tok.split("=", 1)[1]
        elif tok.startswith("gravity"): req["gravity"] = tok.split("=", 1)[1]
        elif tok.startswith("resize"): req["resize"] = tok.split("=", 1)[1]
        elif tok.startswith("format"): fmt = tok.split("=", 1)[1]
        elif tok.startswith("filter"): req["filters"].append(tok.split("-", 1)[1])
    req["flatten"] = (fmt == "jpg")
    return req


# gradmap LUT tails the reference leaves uninitialised (SURVEY App. C-4): no golden case uses 4/6/7/8 colours.
VIGNETTE_TOL = 1   # <= 1 LSB where libm's and CUDA's double cos may differ (DESIGN.md §Exactness)


IO_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_io_v1.npz")


def load_io():
    """tests/golden/golden_io_v1.npz (made by tests/golden/make_golden_io.py from the reference's advancedio.c).
    Returns dict(gifs=[dict(cw, ch, frames=[dict(indices top-down, palette, left, top, dispose, key)], out={0: [...], 1: [...]})],
                 packs=[dict(img, fi24, fi32)], jobs=[dict(gif, query, out)])."""
    z = np.load(IO_PATH)
    meta = json.loads(bytes(z["meta"]).decode())
    gifs = []
    for gi, m in enumerate(meta["gifs"]):
        frames = [dict(f, indices=z[f"g{gi}_idx{fi}"], palette=z[f"g{gi}_pal{fi}"]) for fi, f in enumerate(m["frames"])]
        out = {d: [z[f"g{gi}_d{d}_out{fi}"] for fi in range(len(frames))] for d in (0, 1)}
        gifs.append(dict(cw=m["cw"], ch=m["ch"], frames=frames, out=out))
    packs = [dict(img=z[f"p{pi}_in"], fi24=z[f"p{pi}_fi24"], fi32=z[f"p{pi}_fi32"]) for pi in range(len(meta["packs"]))]
    jobs = [dict(j, out=z[f"j{ji}_out"]) for ji, j in enumerate(meta["jobs"])]
    return dict(gifs=gifs, packs=packs, jobs=jobs)


CV2_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_cv2_v1.json")


def digest(a):
    """SHA-256 of an array's shape and bytes: what golden_cv2_v1.json stores instead of the arrays themselves."""
    a = np.ascontiguousarray(a)
    return hashlib.sha256(repr(a.shape).encode() + a.tobytes()).hexdigest()


def load_cv2():
    """tests/golden/golden_cv2_v1.json (made by tests/golden/make_golden_cv2.py with cv2 4.13, IPP off):
    {case key: {"in": digest of the input, "out": digest of cv2's result}} for the cases below."""
    with open(CV2_PATH) as f:
        return json.load(f)["cases"]


def _rnd(seed, h, w, c):
    return np.random.default_rng(seed).integers(0, 256, (h, w, c), dtype=np.uint8)


def cv2_resize_cases():
    """Random sizes, channel counts and the four interpolations (0 NN, 1 LINEAR, 2 CUBIC, 3 AREA shrink only):
    yields (key, img, dw, dh, mode)."""
    rng = np.random.default_rng(42)
    for it in range(120):
        sw, sh = int(rng.integers(1, 90)), int(rng.integers(1, 70))
        dw, dh = int(rng.integers(1, 120)), int(rng.integers(1, 100))
        c = int(rng.choice([1, 3, 4]))
        img = rng.integers(0, 256, (sh, sw, c), dtype=np.uint8)
        for mode in (0, 1, 2, 3):
            if mode == 3 and (dw > sw or dh > sh):
                continue
            yield f"resize/{it}/{mode}", img, dw, dh, mode


GAUSS_SIGMAS = [0.3, 0.5, 0.8, 1.0, 1.5, 2.0, 2.3, 3.0, 4.7, 6.0, 12.0]


def cv2_gaussian_cases():
    """cvSmooth's Gaussian (BORDER_REPLICATE, sigma as the reference's float): yields (key, img, sigma)."""
    for sigma in GAUSS_SIGMAS:
        for (w, h, c) in [(64, 48, 3), (33, 17, 4), (5, 4, 3), (1, 1, 4)]:
            yield f"gaussian/{sigma}/{w}x{h}x{c}", _rnd(int(sigma * 100) + w, h, w, c), sigma


def cv2_orient_image():
    """The input of the flip / transpose / rotate cases: keys flip/0, flip/1, flip/-1, transpose, rotate90."""
    return _rnd(3, 13, 9, 3)


def fi_page(frame):
    """A golden GIF frame as FreeImage holds the locked page (what LoadGIF reads and the C ABI takes): bottom-up scanlines
    padded to 4 bytes with zeros, plus the true width."""
    idx = np.ascontiguousarray(frame["indices"], np.uint8)
    h, w = idx.shape
    bits = np.zeros((h, (w + 3) & ~3), np.uint8)
    bits[:, :w] = idx[::-1]
    return dict(indices=bits, width=w, palette=frame["palette"], left=frame["left"], top=frame["top"], dispose=frame["dispose"], key=frame["key"])
