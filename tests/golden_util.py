"""Loads tests/golden/golden_v1.npz (made by tests/golden/make_golden.py from the compiled reference + cv2)."""
import ctypes as C
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


# ---- vignette: exact except at pixels whose mask rounding is ambiguous (tests/vignette_ref.py) -----------------------
_HOSTSIM = []


def _hostsim():
    if not _HOSTSIM:
        from conftest import HostSim
        _HOSTSIM.append(HostSim())
    return _HOSTSIM[0]


def vignette_ops(shape, cfgkw, req, must_plan=True):
    """The planner's vignette ops of a request on an h x w x c source, in order, as dicts: cx, cy, the op's frame w, h,
    its table's nx, ny (0: evaluated per pixel), maxr, intensity (through tests/hostsim, hostsim_vignette_ops). A request
    the planner refuses fails, or gives [] when must_plan is False."""
    hs = _hostsim()
    lib = hs.lib
    lib.hostsim_vignette_ops.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_float), C.c_int]
    h, w = shape[0], shape[1]
    c = shape[2] if len(shape) == 3 else 1
    ccfg, k1 = hs.api.Config(**cfgkw).to_c()
    creq, k2 = hs.api.make_request(**req)
    plan, step = C.c_void_p(), C.c_int(-1)
    rc = lib.hostsim_plan_create(C.byref(creq), C.byref(ccfg), w, h, c, C.byref(plan), C.byref(step))
    if rc and not must_plan:
        return []
    assert rc == 0, (req, rc)
    try:
        cap = 64
        iv, fv = (C.c_int * (8 * cap))(), (C.c_float * (2 * cap))()
        n = lib.hostsim_vignette_ops(plan, iv, fv, cap)
        assert n <= cap
        return [dict(cx=iv[8 * k], cy=iv[8 * k + 1], w=iv[8 * k + 2], h=iv[8 * k + 3], nx=iv[8 * k + 4], ny=iv[8 * k + 5],
                     maxr=np.float32(fv[2 * k]), intensity=np.float32(fv[2 * k + 1])) for k in range(n)]
    finally:
        lib.hostsim_plan_destroy(plan)


# Filters that neither move nor mix pixels, and the orientations, which move them without mixing: after the last vignette
# only these let an ambiguous mask entry be traced to the output pixels it can touch.
PER_PIXEL = {"modulate", "colorize", "gamma", "contrast", "gradmap", "vignette", "gotham", "lomo", "kelvin", "rainbow", "scanline"}
ORIENT = {"flip", "rotate"}

# Requests whose vignette frames hold an ambiguous entry but whose later steps mix or reorder pixels in ways the ambiguous
# pixels cannot be traced through (blur, packed bottom-up output): {repr(label): ambiguous entries}. They keep the bound
# of one LSB at under 1 in 1000 bytes. For the fixed seeds and shapes of the suite no such request exists.
UNMAPPED_AMBIGUOUS = {}


def _name(f):
    return f.split("=", 1)[0]


def vignette_allowance(shape, cfgkw, req, out_shape):
    """None when every vignette frame of the request is free of ambiguous entries (the result must be exact). Else a
    boolean image of out_shape[:2], the output pixels an ambiguous entry can reach, or the string "unmapped" when later
    steps mix pixels. Also returns the number of ambiguous table entries."""
    import vignette_ref as VR
    from oracle import oracle as O
    ops = vignette_ops(shape, cfgkw, req)
    filters = req.get("filters", []) or []
    at = [k for k, f in enumerate(filters) if _name(f) == "vignette"]
    assert len(at) == len(ops), (req, len(at), len(ops))
    allowed, n_amb, unmapped = None, 0, False
    for k, op in zip(at, ops):
        nx, ny = VR.table_dims(op["w"], op["h"], op["cx"], op["cy"])
        n = VR.classify(op["maxr"], op["intensity"], nx, ny).count
        if not n:
            continue
        n_amb += n
        rest = filters[k + 1:]
        if req.get("pack") or any(_name(f) not in PER_PIXEL | ORIENT for f in rest):
            unmapped = True
            continue
        _, amb = VR.frame_mask(op)
        img = np.repeat(amb[:, :, None].astype(np.uint8) * 255, 3, axis=2)
        for f in rest:
            if _name(f) in ORIENT:
                code, img = O.apply_filter(img, f, True)
                assert code == 0, f
        assert img.shape[:2] == tuple(out_shape[:2]), (req, img.shape, out_shape)
        allowed = (img[:, :, 0] > 0) if allowed is None else allowed | (img[:, :, 0] > 0)
    if unmapped:
        return "unmapped", n_amb
    return allowed, n_amb


# what the allowance was used for over the session: [(label, ambiguous entries, bytes that differed)]
VIGNETTE_ALLOWANCE_USED = []


def assert_vignette_exact(out, ref, shape, cfgkw, req, label):
    """A result of a request with vignette ops against the oracle's (or the reference mask's): exact, except by at most 1
    at output pixels an ambiguous mask entry reaches (tests/vignette_ref.py). shape: the request's source h, w[, c]."""
    assert out.shape == ref.shape, (label, out.shape, ref.shape)
    d = np.abs(out.astype(int) - ref.astype(int))
    allowed, n_amb = vignette_allowance(shape, cfgkw, req, out.shape)
    if allowed is None:
        assert d.max() == 0, (label, int(d.max()), int((d > 0).sum()), d.size)
        return
    if isinstance(allowed, str):
        assert UNMAPPED_AMBIGUOUS.get(repr(label)) == n_amb, (label, n_amb)
        assert d.max() <= 1 and (d > 0).mean() < 1e-3, (label, int(d.max()), float((d > 0).mean()))
    else:
        assert d.max() <= 1 and d[~allowed].max(initial=0) == 0, (label, int(d.max()), int((d[~allowed] > 0).sum()))
    VIGNETTE_ALLOWANCE_USED.append((repr(label), n_amb, int((d > 0).sum())))


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
