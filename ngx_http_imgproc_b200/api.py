"""
ctypes binding of libimp_gpu.so (include/imp_gpu.h) — the call a user of the reference's operator
layer makes, from Python. Used by tests/ and bench.py; it adds no arithmetic of its own.

The library is the product: if it is missing, cannot be loaded, or no B200 is visible, everything
here raises. There is no CPU path.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np

from . import build as _build

IMP_OK = 0
IMP_ERROR_INVALID_ARGS = 50
IMP_ERROR_NO_SUCH_FILTER = 52
IMP_ERROR_NO_SUCH_WATERMARK = 53
IMP_ERROR_TOO_BIG_TARGET = 54
IMP_ERROR_TOO_MUCH_FILTERS = 55
IMP_ERROR_GPU = 100
INTERP_REFERENCE, INTERP_LINEAR = 0, 1


class CWatermark(C.Structure):
    _fields_ = [("pixels", C.c_void_p), ("width", C.c_int), ("height", C.c_int), ("channels", C.c_int),
                ("step", C.c_int), ("gravity_x", C.c_char), ("gravity_y", C.c_char),
                ("offset_x", C.c_int), ("offset_y", C.c_int), ("opacity", C.c_int)]


class CGifFrame(C.Structure):
    _fields_ = [("indices", C.c_void_p), ("pitch", C.c_int), ("width", C.c_int), ("height", C.c_int), ("left", C.c_int), ("top", C.c_int),
                ("dispose", C.c_int), ("transparency_key", C.c_int), ("palette", C.c_void_p)]


class CConfig(C.Structure):
    _fields_ = [("max_target_w", C.c_uint), ("max_target_h", C.c_uint), ("max_filters", C.c_int),
                ("allow_experiments", C.c_int), ("watermark", C.POINTER(CWatermark))]


class CRequest(C.Structure):
    _fields_ = [("crop", C.c_char_p), ("gravity", C.c_char_p), ("resize", C.c_char_p),
                ("filters", C.POINTER(C.c_char_p)), ("filter_count", C.c_int),
                ("simple_resize", C.c_int), ("flatten", C.c_int), ("interp", C.c_int), ("pack", C.c_int)]


@dataclass
class Config:
    """The Config fields the hot path reads (required.h:110-120), with module.c:117-190's defaults."""
    max_w: int = 2000
    max_h: int = 2000
    max_filters: int = 5
    allow_experiments: bool = False
    watermark: Optional[np.ndarray] = None      # decoded overlay, HxWx{3,4} uint8
    wm_gravity_x: str = "l"
    wm_gravity_y: str = "t"
    wm_offset_x: int = 0
    wm_offset_y: int = 0
    wm_opacity: int = 100

    def to_c(self):
        keep = []
        c = CConfig(self.max_w, self.max_h, self.max_filters, 1 if self.allow_experiments else 0, None)
        if self.watermark is not None:
            wm = np.ascontiguousarray(self.watermark, dtype=np.uint8)
            w = CWatermark(wm.ctypes.data, wm.shape[1], wm.shape[0], wm.shape[2], wm.strides[0],
                           self.wm_gravity_x.encode(), self.wm_gravity_y.encode(), self.wm_offset_x, self.wm_offset_y, self.wm_opacity)
            keep += [wm, w]
            c.watermark = C.pointer(w)
        keep.append(c)
        return c, keep


def make_request(crop=None, gravity=None, resize=None, filters: Sequence[str] = (), simple=False, flatten=False, interp=0, pack=0):
    keep = []
    enc = lambda s: None if s is None else s.encode("latin-1")
    arr = (C.c_char_p * max(1, len(filters)))(*[enc(f) for f in filters])
    keep.append(arr)
    r = CRequest(enc(crop), enc(gravity), enc(resize), arr, len(filters), 1 if simple else 0, 1 if flatten else 0, interp, pack)
    keep.append(r)
    return r, keep


class ImpError(RuntimeError):
    def __init__(self, code, step=None, msg=""):
        super().__init__(f"IMP code {code} step {step} {msg}")
        self.code, self.step = code, step


class Library:
    """libimp_gpu.so loaded through ctypes."""

    def __init__(self, path: Optional[str] = None):
        path = path or _build.LIB
        if not os.path.exists(path):
            raise RuntimeError(f"{path} is missing: run `python -m ngx_http_imgproc_b200.build` "
                               "(nvcc, sm_100a). There is no CPU fallback.")
        self.path = path
        L = self.lib = C.CDLL(path)
        L.imp_gpu_last_error.restype = C.c_char_p
        L.imp_gpu_launch_count.restype = C.c_ulonglong
        L.imp_gpu_plan_algorithmic_bytes.restype = C.c_ulonglong
        L.imp_gpu_plan_algorithmic_bytes.argtypes = [C.c_void_p]
        L.imp_gpu_batch_algorithmic_bytes.restype = C.c_ulonglong
        L.imp_gpu_batch_algorithmic_bytes.argtypes = [C.c_void_p]
        L.imp_gpu_plan_create.argtypes = [C.POINTER(CRequest), C.POINTER(CConfig), C.c_int, C.c_int, C.c_int,
                                          C.POINTER(C.c_void_p), C.POINTER(C.c_int)]
        L.imp_gpu_plan_destroy.argtypes = [C.c_void_p]
        L.imp_gpu_plan_output.argtypes = [C.c_void_p] + [C.POINTER(C.c_int)] * 3
        L.imp_gpu_plan_source_window.argtypes = [C.c_void_p] + [C.POINTER(C.c_int)] * 4
        L.imp_gpu_plan_passes.argtypes = [C.c_void_p]
        L.imp_gpu_run_host.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        L.imp_gpu_run_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
        L.imp_gpu_batch_create.argtypes = [C.POINTER(C.c_void_p)]
        L.imp_gpu_batch_destroy.argtypes = [C.c_void_p]
        L.imp_gpu_batch_clear.argtypes = [C.c_void_p]
        L.imp_gpu_batch_add.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        L.imp_gpu_batch_launch.argtypes = [C.c_void_p, C.c_void_p]
        L.imp_gpu_batch_size.argtypes = [C.c_void_p]
        L.imp_gpu_batch_launches_per_run.argtypes = [C.c_void_p]
        L.imp_gpu_batch_run_host.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.imp_gpu_farm_run_host.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        L.imp_gpu_farm_run_host_policy.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.imp_gpu_batch_submit_host.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]
        L.imp_gpu_batch_wait.argtypes = [C.c_void_p]
        L.imp_gpu_batch_poll.argtypes = [C.c_void_p]
        L.imp_gpu_worker_device.argtypes = [C.c_int, C.c_int, C.c_char_p, C.POINTER(C.c_int)]
        L.imp_gpu_init_worker.argtypes = [C.c_int, C.POINTER(C.c_int)]
        L.imp_gpu_upload_watermark.argtypes = [C.POINTER(CWatermark)]
        L.imp_gpu_plan_cache_stats.argtypes = [C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong), C.POINTER(C.c_int)]
        L.imp_gpu_plan_cache_stats.restype = None
        L.imp_gpu_plan_cache_clear.restype = None
        L.imp_gpu_malloc.argtypes = [C.POINTER(C.c_void_p), C.c_size_t]
        L.imp_gpu_free.argtypes = [C.c_void_p]
        L.imp_gpu_malloc_pitch.argtypes = [C.POINTER(C.c_void_p), C.POINTER(C.c_int), C.c_int, C.c_int]
        L.imp_gpu_host_alloc.argtypes = [C.POINTER(C.c_void_p), C.c_size_t]
        L.imp_gpu_host_free.argtypes = [C.c_void_p]
        L.imp_gpu_upload_2d.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]
        L.imp_gpu_download_2d.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]
        L.imp_gpu_sync.argtypes = [C.c_void_p]
        L.imp_gpu_brightness_host.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float)]
        L.imp_gpu_brightness_device.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float), C.c_void_p]
        L.imp_gpu_ascii_length.restype = C.c_long
        L.imp_gpu_ascii_length.argtypes = [C.c_int, C.c_int]
        L.imp_gpu_batch_brightness_host.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.imp_gpu_batch_ascii_host.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]

    # ---- lifetime ---------------------------------------------------------------------------------
    def last_error(self) -> str:
        return (self.lib.imp_gpu_last_error() or b"").decode()

    def check(self, rc, step=None):
        if rc != IMP_OK:
            raise ImpError(rc, step, self.last_error() if rc == IMP_ERROR_GPU else "")

    def init(self, device: int = 0):
        self.check(self.lib.imp_gpu_init(device))

    def set_device(self, device: int):
        self.check(self.lib.imp_gpu_set_device(device))

    def worker_device(self, worker: int, n_devices: int, spec: Optional[str] = None) -> int:
        """imp_gpu_worker_device: the device worker `worker` takes from `spec` (IMP_GPU_DEVICES's syntax; None or "" =
        0..n_devices-1). Host logic only; raises ImpError (with the offending entry) on a bad list."""
        d = C.c_int(-1)
        rc = self.lib.imp_gpu_worker_device(worker, n_devices, None if spec is None else spec.encode(), C.byref(d))
        if rc != IMP_OK:
            raise ImpError(rc, None, self.last_error())
        return d.value

    def init_worker(self, worker: int) -> int:
        """imp_gpu_init_worker: OnEnvStart of worker `worker` (IMP_GPU_DEVICES from the environment); returns the device."""
        d = C.c_int(-1)
        rc = self.lib.imp_gpu_init_worker(worker, C.byref(d))
        if rc != IMP_OK:
            raise ImpError(rc, None, self.last_error())
        return d.value

    def shutdown(self):
        self.lib.imp_gpu_shutdown()

    def device_count(self) -> int:
        return self.lib.imp_gpu_device_count()

    def launch_count(self) -> int:
        return int(self.lib.imp_gpu_launch_count())

    def upload_watermark(self, cfg: "Config"):
        """imp_gpu_upload_watermark: register the config's overlay and upload it to the current device (once)."""
        ccfg, keep = cfg.to_c()
        self.check(self.lib.imp_gpu_upload_watermark(ccfg.watermark))

    def plan_cache_stats(self):
        h, m, n = C.c_ulonglong(), C.c_ulonglong(), C.c_int()
        self.lib.imp_gpu_plan_cache_stats(C.byref(h), C.byref(m), C.byref(n))
        return dict(hits=int(h.value), misses=int(m.value), entries=n.value)

    def plan_cache_clear(self):
        self.lib.imp_gpu_plan_cache_clear()

    def ascii(self, img: np.ndarray, args: str = "") -> bytes:
        """ASCII (filters.c:486-522) of a host frame."""
        img = np.ascontiguousarray(img if img.ndim == 3 else img[:, :, None], dtype=np.uint8)
        self.lib.imp_gpu_ascii_length.restype = C.c_long
        n = self.lib.imp_gpu_ascii_length(img.shape[1], img.shape[0])
        out = C.create_string_buffer(n + 1)
        self.lib.imp_gpu_ascii_host.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_char_p, C.c_void_p, C.c_long]
        self.check(self.lib.imp_gpu_ascii_host(img.ctypes.data, img.strides[0], img.shape[1], img.shape[0], img.shape[2], args.encode(), out, n))
        return out.raw[:n]

    @staticmethod
    def gif_pages(frames):
        """ctypes array of imp_gpu_gif_frame from dicts: indices (HxW uint8, bottom-up; or H x pitch with `width`: the page as FreeImage pads it), left, top, dispose, key, palette (256x4). Returns (array, keep-alive list)."""
        keep, arr = [], (CGifFrame * len(frames))()
        for i, f in enumerate(frames):
            idx = np.ascontiguousarray(f["indices"], np.uint8); pal = np.ascontiguousarray(f["palette"], np.uint8)
            keep += [idx, pal]
            arr[i] = CGifFrame(idx.ctypes.data, idx.strides[0], f.get("width") or idx.shape[1], idx.shape[0], f["left"], f["top"], f["dispose"], f["key"], pal.ctypes.data)
        return arr, keep

    def gif_album(self, frames, cw: int, ch: int, destructive: bool, plan: "Plan", outs=None, n_streams: int = 4):
        """imp_gpu_gif_album_run_host: pages up as indices, canvases expanded on the device, `plan` over every frame."""
        return GifAlbumJob(self, frames, cw, ch, destructive, plan, outs).run(self, n_streams)

    def gif_expand(self, frames, cw: int, ch: int, destructive: bool):
        """LoadGIF's canvas expansion (advancedio.c:195-248) on the device; frames as for gif_pages."""
        arr, keep = self.gif_pages(frames)
        outs = [np.zeros((ch, cw, 4), np.uint8) for _ in frames]
        ptrs = (C.c_void_p * len(frames))(*[o.ctypes.data for o in outs])
        self.lib.imp_gpu_gif_expand_host.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int]
        self.check(self.lib.imp_gpu_gif_expand_host(arr, len(frames), cw, ch, 1 if destructive else 0, ptrs, cw * 4))
        return outs

    def brightness(self, img: np.ndarray) -> float:
        """CalcPerceivedBrightness (filters.c:707-729) of a host frame, reduced on the device."""
        img = np.ascontiguousarray(img if img.ndim == 3 else img[:, :, None], dtype=np.uint8)
        out = C.c_float(0)
        self.check(self.lib.imp_gpu_brightness_host(img.ctypes.data, img.strides[0], img.shape[1], img.shape[0], img.shape[2], C.byref(out)))
        return float(out.value)

    # ---- answers instead of frames: format=json / format=text over a batch ----------------------------
    def batch_brightness(self, plans: List["Plan"], srcs: List[np.ndarray], n_streams: int = 4) -> np.ndarray:
        """imp_gpu_batch_brightness_host: job i runs plans[i] on srcs[i]; CalcPerceivedBrightness of each result (float32)."""
        n = len(plans)
        P, S, SS = _job_arrays(plans, srcs)
        out = np.zeros(n, np.float32)
        self.check(self.lib.imp_gpu_batch_brightness_host(n, P, S, SS, out.ctypes.data, n_streams))
        return out

    def batch_ascii(self, plans: List["Plan"], srcs: List[np.ndarray], args=None, n_streams: int = 4) -> List[bytes]:
        """imp_gpu_batch_ascii_host: ASCII of each result. `args`: one value for every job or a list (None: 10-level ramp)."""
        n = len(plans)
        P, S, SS = _job_arrays(plans, srcs)
        args = list(args) if isinstance(args, (list, tuple)) else [args] * n
        A = (C.c_char_p * max(n, 1))(*[None if a is None else a.encode() for a in args])
        lens = [self.lib.imp_gpu_ascii_length(p.out_w, p.out_h) for p in plans]
        bufs = [C.create_string_buffer(max(k, 1)) for k in lens]
        T = (C.c_void_p * max(n, 1))(*[C.addressof(b) for b in bufs])
        caps = (C.c_long * max(n, 1))(*lens)
        self.check(self.lib.imp_gpu_batch_ascii_host(n, P, S, SS, A, T, caps, n_streams))
        return [b.raw[:k] for b, k in zip(bufs, lens)]

    # ---- plans --------------------------------------------------------------------------------------
    def plan(self, w, h, c, cfg: Optional[Config] = None, **req) -> "Plan":
        cfg = cfg or Config()
        ccfg, keep1 = cfg.to_c()
        creq, keep2 = make_request(**req)
        out, step = C.c_void_p(), C.c_int(-1)
        rc = self.lib.imp_gpu_plan_create(C.byref(creq), C.byref(ccfg), w, h, c, C.byref(out), C.byref(step))
        if rc != IMP_OK:
            raise ImpError(rc, step.value)
        return Plan(self, out, (w, h, c))

    def try_plan(self, w, h, c, cfg: Optional[Config] = None, **req):
        """Returns (code, step, plan-or-None) without raising on validation errors."""
        try:
            p = self.plan(w, h, c, cfg, **req)
            return IMP_OK, 8, p
        except ImpError as e:
            return e.code, e.step, None

    # ---- one call: host image in, host image out (the e2e path) ---------------------------------------
    def run(self, img: np.ndarray, cfg: Optional[Config] = None, **req) -> np.ndarray:
        img = np.ascontiguousarray(img if img.ndim == 3 else img[:, :, None], dtype=np.uint8)
        p = self.plan(img.shape[1], img.shape[0], img.shape[2], cfg, **req)
        try:
            return p.run_host(img)
        finally:
            p.close()


class Plan:
    def __init__(self, lib: Library, handle, src_shape):
        self.L, self.h, self.src = lib, handle, src_shape
        w, h, c = C.c_int(), C.c_int(), C.c_int()
        lib.lib.imp_gpu_plan_output(handle, C.byref(w), C.byref(h), C.byref(c))
        self.out_w, self.out_h, self.out_c = w.value, h.value, c.value
        x, y = C.c_int(), C.c_int()
        lib.lib.imp_gpu_plan_source_window(handle, C.byref(x), C.byref(y), C.byref(w), C.byref(h))
        self.window = (x.value, y.value, w.value, h.value)
        self.passes = lib.lib.imp_gpu_plan_passes(handle)
        self.algorithmic_bytes = int(lib.lib.imp_gpu_plan_algorithmic_bytes(handle))

    def close(self):
        if self.h:
            self.L.lib.imp_gpu_plan_destroy(self.h)
            self.h = None

    def run_host(self, img: np.ndarray, out: Optional[np.ndarray] = None) -> np.ndarray:
        img = np.ascontiguousarray(img if img.ndim == 3 else img[:, :, None], dtype=np.uint8)
        assert (img.shape[1], img.shape[0], img.shape[2]) == self.src
        if out is None:
            out = np.empty((self.out_h, self.out_w, self.out_c), np.uint8)
        self.L.check(self.L.lib.imp_gpu_run_host(self.h, img.ctypes.data, img.strides[0], out.ctypes.data, out.strides[0]))
        return out

    def run_device(self, d_src: int, src_pitch: int, d_dst: int, dst_pitch: int, stream: int = 0):
        self.L.check(self.L.lib.imp_gpu_run_device(self.h, d_src, src_pitch, d_dst, dst_pitch, stream))


class Batch:
    def __init__(self, lib: Library):
        self.L = lib
        self.h = C.c_void_p()
        lib.check(lib.lib.imp_gpu_batch_create(C.byref(self.h)))

    def add(self, plan: Plan, d_src: int, src_pitch: int, d_dst: int, dst_pitch: int):
        self.L.check(self.L.lib.imp_gpu_batch_add(self.h, plan.h, d_src, src_pitch, d_dst, dst_pitch))

    def launch(self, stream: int = 0):
        self.L.check(self.L.lib.imp_gpu_batch_launch(self.h, stream))

    def clear(self):
        self.L.lib.imp_gpu_batch_clear(self.h)

    @property
    def algorithmic_bytes(self) -> int:
        return int(self.L.lib.imp_gpu_batch_algorithmic_bytes(self.h))

    @property
    def launches_per_run(self) -> int:
        return self.L.lib.imp_gpu_batch_launches_per_run(self.h)

    def close(self):
        if self.h:
            self.L.lib.imp_gpu_batch_destroy(self.h)
            self.h = None


FARM_ROUND_ROBIN, FARM_SIZE_AWARE = 0, 1


def _job_arrays(plans, srcs):
    n = max(len(plans), 1)
    return ((C.c_void_p * n)(*[p.h for p in plans]), (C.c_void_p * n)(*[s.ctypes.data for s in srcs]),
            (C.c_int * n)(*[s.strides[0] for s in srcs]))


class HostJobs:
    """The five parallel argument arrays of the host-batch entry points, built once (bench loops reuse them)."""

    def __init__(self, plans: List[Plan], srcs: List[np.ndarray], dsts: List[np.ndarray]):
        n = self.n = len(plans)
        self.keep = (plans, srcs, dsts)
        self.P = (C.c_void_p * n)(*[p.h for p in plans])
        self.S = (C.c_void_p * n)(*[s.ctypes.data for s in srcs])
        self.D = (C.c_void_p * n)(*[d.ctypes.data for d in dsts])
        self.SS = (C.c_int * n)(*[s.strides[0] for s in srcs])
        self.DS = (C.c_int * n)(*[d.strides[0] for d in dsts])

    def run(self, lib: Library, n_streams=4, n_gpus=0, policy=FARM_ROUND_ROBIN):
        if n_gpus:
            lib.check(lib.lib.imp_gpu_farm_run_host_policy(self.n, self.P, self.S, self.SS, self.D, self.DS, n_gpus, n_streams, policy))
        else:
            lib.check(lib.lib.imp_gpu_batch_run_host(self.n, self.P, self.S, self.SS, self.D, self.DS, n_streams))

    def submit(self, lib: Library, n_streams=4):
        """imp_gpu_batch_submit_host: returns a ticket for wait()."""
        t = C.c_void_p()
        lib.check(lib.lib.imp_gpu_batch_submit_host(self.n, self.P, self.S, self.SS, self.D, self.DS, n_streams, C.byref(t)))
        return t

    @staticmethod
    def poll(lib: Library, ticket) -> bool:
        return bool(lib.lib.imp_gpu_batch_poll(ticket))

    @staticmethod
    def wait(lib: Library, ticket):
        lib.check(lib.lib.imp_gpu_batch_wait(ticket))


class GifAlbumJob:
    """imp_gpu_gif_album_run_host with its argument arrays built once: `pages` as Library.gif_pages takes them, one plan for
    every frame (a frame whose entry in `plans` is None only takes part in the disposal replay), outputs given or allocated."""

    def __init__(self, lib: Library, pages, cw: int, ch: int, destructive: bool, plans, outs=None):
        n = self.n = len(pages)
        plans = list(plans) if isinstance(plans, (list, tuple)) else [plans] * n
        self.arr, self.keep = Library.gif_pages(pages)
        if outs is None:
            outs = [None if p is None else np.empty((p.out_h, p.out_w, p.out_c), np.uint8) for p in plans]
        self.outs, self.plans = outs, plans
        self.P = (C.c_void_p * n)(*[None if p is None else p.h for p in plans])
        self.D = (C.c_void_p * n)(*[None if o is None else o.ctypes.data for o in outs])
        self.DS = (C.c_int * n)(*[0 if o is None else o.strides[0] for o in outs])
        self.geom = (cw, ch, 1 if destructive else 0)
        self.h2d_bytes = sum(int(np.asarray(f["indices"]).size) + 1024 for f in pages)
        self.d2h_bytes = sum(0 if p is None else p.out_w * p.out_h * p.out_c for p in plans)
        self.out_pixels = sum(0 if p is None else p.out_w * p.out_h for p in plans)
        lib.lib.imp_gpu_gif_album_run_host.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]

    def run(self, lib: Library, n_streams=4):
        cw, ch, d = self.geom
        lib.check(lib.lib.imp_gpu_gif_album_run_host(self.arr, self.n, cw, ch, d, self.P, self.D, self.DS, n_streams))
        return self.outs


def farm_assign(lib: Library, plans: List[Plan], n_gpus: int, policy=FARM_ROUND_ROBIN) -> List[int]:
    """imp_gpu_farm_assign: the GPU each job would run on (host logic only; works without a device)."""
    n = len(plans)
    P = (C.c_void_p * max(n, 1))(*[p.h for p in plans])
    owner = (C.c_int * max(n, 1))()
    lib.lib.imp_gpu_farm_assign.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    lib.check(lib.lib.imp_gpu_farm_assign(n, P, n_gpus, policy, owner))
    return list(owner[:n])


def run_host_batch(lib: Library, plans: List[Plan], srcs: List[np.ndarray], dsts: List[np.ndarray], n_streams=4, n_gpus=0, policy=FARM_ROUND_ROBIN):
    """imp_gpu_batch_run_host / imp_gpu_farm_run_host[_policy] over numpy (or pinned) buffers."""
    HostJobs(plans, srcs, dsts).run(lib, n_streams, n_gpus, policy)


# ---- the reference-signature operator layer (include/imp_ops.h) -----------------------------------------------------
class IplROI(C.Structure):
    _fields_ = [("coi", C.c_int), ("xOffset", C.c_int), ("yOffset", C.c_int), ("width", C.c_int), ("height", C.c_int)]


class IplImage(C.Structure):
    """OpenCV 2.4 types_c.h layout (sizeof == 144 on x86-64), as include/imp_ops.h declares it."""
    pass


IplImage._fields_ = [("nSize", C.c_int), ("ID", C.c_int), ("nChannels", C.c_int), ("alphaChannel", C.c_int), ("depth", C.c_int),
                     ("colorModel", C.c_char * 4), ("channelSeq", C.c_char * 4), ("dataOrder", C.c_int), ("origin", C.c_int),
                     ("align", C.c_int), ("width", C.c_int), ("height", C.c_int), ("roi", C.POINTER(IplROI)),
                     ("maskROI", C.POINTER(IplImage)), ("imageId", C.c_void_p), ("tileInfo", C.c_void_p), ("imageSize", C.c_int),
                     ("imageData", C.c_void_p), ("widthStep", C.c_int), ("BorderMode", C.c_int * 4), ("BorderConst", C.c_int * 4),
                     ("imageDataOrigin", C.c_void_p)]


class OpsLayer:
    """imp_Crop / imp_Resize / imp_Filter / imp_Watermark / imp_BlendWithPaper / imp_FlushAll driven the way RunJob's
    loops (bridge.c:574-656) drive the reference's operators: record + validate per operator, one fused flush."""
    CREATE_T = C.CFUNCTYPE(C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int)
    RELEASE_T = C.CFUNCTYPE(None, C.POINTER(C.c_void_p))

    def __init__(self, lib: Library):
        self.L = lib
        L = lib.lib
        PP = C.POINTER(C.POINTER(IplImage))
        L.imp_Crop.argtypes = [PP, C.c_char_p, C.c_char_p]
        L.imp_Resize.argtypes = [PP, C.c_char_p, C.POINTER(CConfig), C.c_int]
        L.imp_Filter.argtypes = [PP, C.c_char_p, C.c_int]
        L.imp_Watermark.argtypes = [C.POINTER(IplImage), C.POINTER(CConfig)]
        L.imp_BlendWithPaper.argtypes = [C.POINTER(IplImage)]
        L.imp_FlushAll.argtypes = [PP, C.c_int]
        L.imp_FlushAllGif.argtypes = [PP, C.c_int, C.c_void_p, C.c_int, C.c_int]
        L.imp_Discard.argtypes = [C.POINTER(IplImage)]
        L.imp_Brightness.argtypes = [C.POINTER(IplImage), C.POINTER(C.c_float)]
        L.imp_Ascii.argtypes = [C.POINTER(IplImage), C.c_char_p, C.c_void_p, C.c_long]
        L.imp_ops_pending.argtypes = [C.POINTER(IplImage)]
        self.keep = []
        self._cb = (self.CREATE_T(self._create), self.RELEASE_T(self._release))
        L.imp_ops_set_image_allocator.argtypes = [self.CREATE_T, self.RELEASE_T]
        L.imp_ops_set_image_allocator(*self._cb)

    @staticmethod
    def header(img: np.ndarray):
        """IplImage header over `img` (H x W x C uint8, C-contiguous rows; widthStep = its row stride)."""
        h, w, c = img.shape
        im = IplImage()
        im.nSize = C.sizeof(IplImage); im.nChannels = c; im.depth = 8; im.width = w; im.height = h; im.align = 4
        im.widthStep = img.strides[0]; im.imageSize = img.strides[0] * h
        im.imageData = img.ctypes.data; im.imageDataOrigin = img.ctypes.data
        return im

    def _create(self, w, h, depth, c):
        step = (w * c + 3) & ~3
        buf = np.empty((h, step), np.uint8)
        im = IplImage()
        im.nSize = C.sizeof(IplImage); im.nChannels = c; im.depth = depth; im.width = w; im.height = h; im.align = 4
        im.widthStep = step; im.imageSize = step * h
        im.imageData = buf.ctypes.data; im.imageDataOrigin = buf.ctypes.data
        self.keep.append((im, buf))
        return C.addressof(im)

    def _release(self, pp):
        pp[0] = None

    def record(self, frames, cfg: Config, crop=None, gravity=None, resize=None, filters=(), simple=False, flatten=False):
        """The per-frame operator calls of RunJob (bridge.c:576-656) over `frames` (numpy images), nothing run yet.
        Returns (code, IplImage pointers or None); on an error everything recorded is discarded."""
        L = self.L.lib
        self.keep = []
        ccfg, keep = cfg.to_c()
        enc = lambda t: None if t is None else t.encode("latin-1")
        ptrs = [C.pointer(self.header(f)) for f in frames]
        code = 0
        for p in ptrs:
            if crop is not None and not code: code = L.imp_Crop(C.byref(p), enc(crop), enc(gravity))
            if resize is not None and not code: code = L.imp_Resize(C.byref(p), enc(resize), C.byref(ccfg), 1 if simple else 0)
            for f in filters:
                if not code: code = L.imp_Filter(C.byref(p), enc(f), 1 if cfg.allow_experiments else 0)
            if cfg.watermark is not None and not code: code = L.imp_Watermark(p, C.byref(ccfg))
            if flatten and not code: code = L.imp_BlendWithPaper(p)
        if code:
            for p in ptrs: L.imp_Discard(p)
            return code, None
        return 0, ptrs

    def brightness(self, frames, cfg: Config, **req):
        """Records like request() and returns (code, [imp_Brightness of each frame] or None); the recording is then discarded."""
        code, ptrs = self.record(frames, cfg, **req)
        if code:
            return code, None
        out, v = [], C.c_float()
        for p in ptrs:
            if not code:
                code = self.L.lib.imp_Brightness(p, C.byref(v))
                out.append(float(v.value))
            self.L.lib.imp_Discard(p)
        return (code, None) if code else (0, out)

    def ascii(self, frames, cfg: Config, args=None, **req):
        """Records like request() and returns (code, [imp_Ascii of each frame] or None); the recording is then discarded."""
        code, ptrs = self.record(frames, cfg, **req)
        if code:
            return code, None
        out = []
        for p in ptrs:
            if not code:
                im = p.contents                                          # the header describes the result the flush would leave
                w, h = (im.width, im.height)
                n = self.L.lib.imp_gpu_ascii_length(w, h)
                buf = C.create_string_buffer(max(n, 1))
                code = self.L.lib.imp_Ascii(p, None if args is None else args.encode(), buf, n)
                out.append(buf.raw[:n])
            self.L.lib.imp_Discard(p)
        return (code, None) if code else (0, out)

    def request(self, frames, cfg: Config, crop=None, gravity=None, resize=None, filters=(), simple=False, flatten=False, gif_pages=None, destructive=False):
        """Steps 3-7 of RunJob over `frames` (numpy images): returns (code, list of results or None).
        gif_pages (dicts as Library.gif_pages takes them): `frames` are only canvas-sized 4-channel placeholders whose pixels
        are never read; the flush is imp_FlushAllGif (pages expanded on the device)."""
        L = self.L.lib
        code, ptrs = self.record(frames, cfg, crop, gravity, resize, filters, simple, flatten)
        if code:
            return code, None
        arr = (C.POINTER(IplImage) * len(ptrs))(*ptrs)
        if gif_pages is not None:
            pages, keep_pages = Library.gif_pages(gif_pages)
            code = L.imp_FlushAllGif(arr, len(ptrs), pages, len(gif_pages), 1 if destructive else 0)
        else:
            code = L.imp_FlushAll(arr, len(ptrs))
        if code:
            return code, None
        outs = []
        for k in range(len(ptrs)):
            im = arr[k].contents
            raw = (C.c_ubyte * (im.widthStep * im.height)).from_address(im.imageData)
            a = np.frombuffer(raw, np.uint8).reshape(im.height, im.widthStep)[:, :im.width * im.nChannels]
            outs.append(a.reshape(im.height, im.width, im.nChannels))
        return 0, outs


_default: Optional[Library] = None


def library() -> Library:
    """The process-wide library handle (built on demand when nvcc is present)."""
    global _default
    if _default is None:
        override = os.environ.get("IMP_GPU_LIB")           # A/B tuning: load another build of the same ABI
        if override:
            _default = Library(override)
        else:
            if _build.stale():
                _build.build()
            _default = Library()
    return _default
