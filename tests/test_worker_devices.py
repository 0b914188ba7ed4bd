"""Worker placement: which GPU each nginx worker process takes (imp_gpu_worker_device / imp_gpu_init_worker and
IMP_GPU_DEVICES), the drop-in's OnEnvStart that calls it, and the farm following the same device list.

CPU: the mapping, every rejected list, the no-device path, a C99 host, and OnEnvStart compiled against stand-in nginx
headers that record its log lines. GPU: forked workers (the nginx process model) check their device independently of
the returned index, through the CUDA driver, and serve exact requests on it; the farm and the reference's own RunJob
over the drop-in follow the list."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import ngx_http_imgproc_b200 as M
from conftest import ROOT, smooth_image
from ngx_http_imgproc_b200 import api


def _worker_device(L, worker, n, spec):
    d = C.c_int(7)
    rc = L.lib.imp_gpu_worker_device(worker, n, None if spec is None else spec.encode(), C.byref(d))
    return rc, d.value, L.last_error()


# ---- CPU ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("spec", [None, ""])
def test_default_list_maps_worker_modulo_device_count(spec):
    L = M.library()
    for n in (1, 4, 8):
        assert [L.worker_device(k, n, spec) for k in range(18)] == [k % n for k in range(18)]


def test_explicit_list_is_taken_in_order():
    L = M.library()
    assert [L.worker_device(k, 4, "3,1,2") for k in range(6)] == [3, 1, 2, 3, 1, 2]
    assert [L.worker_device(k, 8, "4,0,5,1") for k in range(8)] == [4, 0, 5, 1] * 2
    assert [L.worker_device(k, 2, "1") for k in range(3)] == [1, 1, 1]
    assert L.worker_device(5, 16, ",".join(str(d) for d in range(16))) == 5       # 16 entries: the most a list holds


@pytest.mark.parametrize("spec,n,entry,token", [
    ("a", 4, 1, "a"), ("1,,2", 4, 2, ""), ("0,1,", 4, 3, ""), ("-1", 4, 1, "-1"), ("4", 4, 1, "4"), ("1,1", 4, 2, "1"),
    (",".join(str(d) for d in range(17)), 32, 17, "16"), (" 1", 4, 1, " 1"), (",", 4, 1, ""), ("0,1x", 4, 2, "1x"),
    ("99999999999999999999", 4, 1, "99999999999999999999"), ("16", 32, 1, "16")])
def test_a_bad_list_is_refused_and_names_its_entry(spec, n, entry, token):
    L = M.library()
    rc, d, msg = _worker_device(L, 0, n, spec)
    assert (rc, d) == (M.IMP_ERROR_INVALID_ARGS, -1), (spec, rc, d)
    assert f'entry {entry} ("{token}")' in msg and spec in msg, msg
    with pytest.raises(M.ImpError) as e:
        L.worker_device(0, n, spec)
    assert e.value.code == M.IMP_ERROR_INVALID_ARGS and f'("{token}")' in str(e.value)


def test_negative_worker_and_no_devices():
    L = M.library()
    rc, d, msg = _worker_device(L, -1, 4, None)
    assert (rc, d) == (M.IMP_ERROR_INVALID_ARGS, -1) and "-1" in msg
    rc, d, msg = _worker_device(L, 0, 0, None)
    assert (rc, d) == (M.IMP_ERROR_GPU, -1) and msg
    assert _worker_device(L, 0, -3, "0")[:2] == (M.IMP_ERROR_GPU, -1)
    assert L.lib.imp_gpu_worker_device(0, 4, None, None) == M.IMP_ERROR_INVALID_ARGS


def test_init_worker_without_a_device_initialises_nothing(monkeypatch):
    L = M.library()
    if L.device_count() > 0:
        pytest.skip("a GPU is present")
    for spec in (None, "0", "x"):
        if spec is None:
            monkeypatch.delenv("IMP_GPU_DEVICES", raising=False)
        else:
            monkeypatch.setenv("IMP_GPU_DEVICES", spec)
        d = C.c_int(7)
        assert L.lib.imp_gpu_init_worker(2, C.byref(d)) == M.IMP_ERROR_GPU and d.value == -1
        assert "no CUDA device" in L.last_error()
        with pytest.raises(M.ImpError) as e:
            L.init_worker(2)
        assert e.value.code == M.IMP_ERROR_GPU
        plan = L.plan(8, 8, 3, resize="4,4")
        out = np.full((4, 4, 3), 7, np.uint8)
        with pytest.raises(M.ImpError) as e:
            plan.run_host(np.zeros((8, 8, 3), np.uint8), out)
        assert e.value.code == M.IMP_ERROR_GPU and "has not been called" in str(e.value) and (out == 7).all()
        plan.close()


def test_a_c99_host_maps_workers(tmp_path):
    src = tmp_path / "workers.c"
    src.write_text(r'''
#include <stdio.h>
#include <string.h>
#include "imp_gpu.h"
int main(void) {
    int k, d = 0, expect[6] = {3, 1, 2, 3, 1, 2};
    for (k = 0; k < 6; k++)
        if (imp_gpu_worker_device(k, 4, "3,1,2", &d) != IMP_OK || d != expect[k]) return 1;
    if (imp_gpu_worker_device(9, 4, NULL, &d) != IMP_OK || d != 1) return 2;
    if (imp_gpu_worker_device(0, 4, "1,1", &d) != IMP_ERROR_INVALID_ARGS || d != -1) return 3;
    if (!strstr(imp_gpu_last_error(), "(\"1\")")) return 4;
    if (imp_gpu_worker_device(0, 0, NULL, &d) != IMP_ERROR_GPU) return 5;
    if (imp_gpu_device_count() == 0 && (imp_gpu_init_worker(0, &d) != IMP_ERROR_GPU || d != -1)) return 6;
    printf("WORKERS OK\n");
    return 0;
}
''')
    exe = tmp_path / "workers"
    pkg = os.path.join(ROOT, "ngx_http_imgproc_b200")
    r = subprocess.run(["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src),
                        "-L", pkg, "-limp_gpu", "-Wl,-rpath," + pkg], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0 and "WORKERS OK" in r.stdout, (r.returncode, r.stdout, r.stderr)


# The drop-in compiled as nginx compiles it: its own includes resolve to these stand-ins (ngx_log_error records the line
# instead of being a no-op) and to a required.h that declares only the reference types imp_dropin.c reads.
_NGX_CONFIG = r'''
#ifndef TEST_NGX_CONFIG_H
#define TEST_NGX_CONFIG_H
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <stdint.h>
#include <sys/types.h>
typedef intptr_t ngx_int_t; typedef uintptr_t ngx_uint_t;
typedef struct { size_t len; unsigned char* data; } ngx_str_t;
#define NGX_LOG_EMERG  1
#define NGX_LOG_NOTICE 6
void test_log_line(int level, const char* fmt, ...);
#define ngx_log_error(level, log, err, ...) ((void)(log), (void)(err), test_log_line(level, __VA_ARGS__))
#endif
'''
_NGX_CORE = r'''
#ifndef TEST_NGX_CORE_H
#define TEST_NGX_CORE_H
#include "ngx_config.h"
typedef struct { void* log; } ngx_cycle_t;
extern volatile ngx_cycle_t* ngx_cycle;
extern ngx_uint_t ngx_worker;
#endif
'''
_REQUIRED = r'''
#include "ngx_config.h"
#include <opencv/cv.h>
#define IMP_OK 0
#define IMP_ERROR_MALLOC_FAILED 2
#define IMP_ERROR_INVALID_ARGS 50
typedef struct { char GravityX, GravityY; int OffsetX, OffsetY; } Position;
typedef struct { unsigned W, H; } Dimensions;
typedef struct { CvSize Size; int Depth, Channels, Step; size_t Length; void* Pointer; } RecoverInfo;
typedef struct { ssize_t Enable; size_t MaxSrcSize; ngx_str_t WatermarkPath; ssize_t WatermarkOpacity; Position* WatermarkPosition;
                 RecoverInfo* WatermarkInfo; Dimensions* MaxTargetDimensions; ssize_t MaxFiltersCount; ssize_t AllowExperiments; } Config;
typedef struct { IplImage* Image; int Time, Dispose, TransparencyKey; } Frame;
typedef struct { Frame* Frames; int Count; int Error; } Album;
'''
_MAIN = r'''
#include <stdarg.h>
#include "ngx_core.h"
#include <opencv/cv.h>
#include "imp_gpu.h"
static char test_log[4096];
void test_log_line(int level, const char* fmt, ...) {
    size_t n = strlen(test_log);
    va_list ap;
    n += (size_t)snprintf(test_log + n, sizeof test_log - n, "%d|", level);
    va_start(ap, fmt);
    n += (size_t)vsnprintf(test_log + n, sizeof test_log - n, fmt, ap);
    va_end(ap);
    snprintf(test_log + n, sizeof test_log - n, "\n");
}
static ngx_cycle_t cycle;
volatile ngx_cycle_t* ngx_cycle = &cycle;
ngx_uint_t ngx_worker;
IplImage* cvCreateImage(CvSize s, int depth, int c) { (void)s; (void)depth; (void)c; return NULL; }
void cvReleaseImage(IplImage** p) { (void)p; }
void OnEnvStart(void);
void OnEnvDestroy(void);
int main(int argc, char** argv) {
    ngx_worker = (ngx_uint_t)atoi(argv[1]);
    OnEnvStart();
    printf("%d\n%s", imp_gpu_device_count(), test_log);
    OnEnvDestroy();
    return argc == 2 ? 0 : 1;
}
'''


@pytest.fixture(scope="module")
def onenvstart_host(tmp_path_factory):
    d = tmp_path_factory.mktemp("dropin")
    for name, text in (("ngx_config.h", _NGX_CONFIG), ("ngx_core.h", _NGX_CORE), ("required.h", _REQUIRED), ("main.c", _MAIN),
                       ("bridge.h", ""), ("filters.h", "")):
        (d / name).write_text(text)
    exe = d / "onenvstart"
    pkg = os.path.join(ROOT, "ngx_http_imgproc_b200")
    r = subprocess.run(["gcc", "-Wall", "-Werror", "-I", str(d), "-I", os.path.join(ROOT, "oracle", "shim"), "-I", os.path.join(ROOT, "include"),
                        "-o", str(exe), str(d / "main.c"), os.path.join(pkg, "dropin", "imp_dropin.c"),
                        "-L", pkg, "-limp_gpu", "-Wl,-rpath," + pkg], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return str(exe)


@pytest.mark.parametrize("worker,spec", [(0, None), (3, None), (3, "0"), (1, "x"), (2, "5,5")])
def test_onenvstart_places_the_worker_and_logs_the_outcome(onenvstart_host, worker, spec):
    """One NOTICE line naming worker and GPU, or one EMERG line naming the worker and the library's reason."""
    env = {k: v for k, v in os.environ.items() if k != "IMP_GPU_DEVICES"}
    if spec is not None:
        env["IMP_GPU_DEVICES"] = spec
    r = subprocess.run([onenvstart_host, str(worker)], capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0, r.stderr
    n, *lines = r.stdout.splitlines()
    n = int(n)
    assert len(lines) == 1, lines
    if n == 0:
        assert lines[0].startswith(f"1|imgproc: worker {worker} has no GPU: no CUDA device"), lines
    elif spec in ("x", "5,5"):
        assert lines[0].startswith(f"1|imgproc: worker {worker} has no GPU: device list \"{spec}\""), lines
    else:
        expect = int(spec) if spec else worker % n
        assert lines[0] == f"6|imgproc: worker {worker} on GPU {expect}", lines


def test_dropin_links_without_nginx_and_takes_its_worker_index_from_ngx_worker(tmp_path):
    """Against the oracle's stand-in nginx headers (the reference's test build compiles the drop-in so), nothing defines
    ngx_worker: the drop-in's weak definition does, as worker 0, and a host sets it before OnEnvStart."""
    for name, text in (("required.h", _REQUIRED), ("bridge.h", ""), ("filters.h", ""),
                       ("cv.c", "#include <opencv/cv.h>\nIplImage* cvCreateImage(CvSize s, int d, int c) { (void)s; (void)d; (void)c; return 0; }\n"
                                "void cvReleaseImage(IplImage** p) { (void)p; }\n")):
        (tmp_path / name).write_text(text)
    so = tmp_path / "libdropin.so"
    pkg = os.path.join(ROOT, "ngx_http_imgproc_b200")
    r = subprocess.run(["gcc", "-O1", "-fPIC", "-shared", "-Wall", "-Werror", "-I", str(tmp_path), "-I", os.path.join(ROOT, "oracle", "shim"),
                        "-I", os.path.join(ROOT, "include"), "-o", str(so), os.path.join(pkg, "dropin", "imp_dropin.c"), str(tmp_path / "cv.c"),
                        "-L", pkg, "-limp_gpu", "-Wl,-rpath," + pkg], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lib = C.CDLL(str(so))
    w = C.c_size_t.in_dll(lib, "ngx_worker")
    assert w.value == 0
    w.value = 5
    assert C.c_size_t.in_dll(C.CDLL(str(so)), "ngx_worker").value == 5


# ---- GPU ------------------------------------------------------------------------------------------------------------
_CUDA_DRIVER = r"""
import ctypes as C
def _cu():                                   # only after the library created its context: cuInit before fork() would poison the workers
    cu = C.CDLL("libcuda.so.1")
    assert cu.cuInit(0) == 0
    return cu
def pointer_device(p):
    v = C.c_int(-1)
    assert _cu().cuPointerGetAttribute(C.byref(v), 9, C.c_void_p(p)) == 0      # CU_POINTER_ATTRIBUTE_DEVICE_ORDINAL
    return v.value
def current_device():
    v = C.c_int(-1)
    assert _cu().cuCtxGetDevice(C.byref(v)) == 0
    return v.value
def context_active(ordinal):
    cu, dev, flags, active = _cu(), C.c_int(), C.c_uint(), C.c_int()
    assert cu.cuDeviceGet(C.byref(dev), ordinal) == 0
    assert cu.cuDevicePrimaryCtxGetState(dev, C.byref(flags), C.byref(active)) == 0
    return bool(active.value)
"""

# A master process that loads the library and validates requests without initialising CUDA, then forks one process per
# worker, as nginx does. argv: spec ("-" = IMP_GPU_DEVICES unset), then the device each worker must land on (-1: the list
# is bad and the worker must get no device).
_WORKERS = r"""
import json, os, sys, ctypes as C, numpy as np
sys.path.insert(0, "."); sys.path.insert(0, "tests")
import ngx_http_imgproc_b200 as M
from ngx_http_imgproc_b200 import api
from oracle import oracle as O
from conftest import smooth_image
DRIVER
spec, expect = sys.argv[1], json.loads(sys.argv[2])
if spec == "-": os.environ.pop("IMP_GPU_DEVICES", None)
else: os.environ["IMP_GPU_DEVICES"] = spec
L = M.library()
wm = smooth_image(9, 10, 14, 4)
kw = dict(max_w=0, max_h=0, allow_experiments=True, watermark=wm, wm_gravity_x="r", wm_gravity_y="b", wm_offset_x=2, wm_offset_y=1, wm_opacity=70)
cfg = api.Config(**kw)
img, img2 = smooth_image(1, 240, 320, 4), smooth_image(2, 90, 130, 3)
rq = dict(crop="300px,200px,c,c", resize="150,100", filters=["gamma=1.2", "rotate=90"])
rq2 = dict(resize="61,37", filters=["modulate=10,90,100"])
orc = lambda im, r: O.run_chain(im, r.get("crop"), None, r.get("resize"), r.get("filters"), O.OracleConfig(**kw))[2]
ref, ref2 = orc(img, rq), orc(img2, rq2)
assert L.try_plan(64, 48, 3, cfg, resize="0,0")[0] == 50     # the master validates; CUDA is not touched before fork
pids = []
for k, want in enumerate(expect):
    pid = os.fork()
    if pid == 0:
        try:
            if want < 0:
                try:
                    L.init_worker(k); raise AssertionError("init_worker accepted a bad list")
                except M.ImpError as e:
                    assert e.code == M.IMP_ERROR_INVALID_ARGS and spec in str(e), e
                p = L.plan(320, 240, 4, cfg, **rq)
                out = np.full((p.out_h, p.out_w, p.out_c), 7, np.uint8)
                try:
                    p.run_host(img, out); raise AssertionError("a run without a device succeeded")
                except M.ImpError as e:
                    assert e.code == M.IMP_ERROR_GPU, e
                dst = out.copy()
                assert L.lib.imp_gpu_batch_run_host(1, (C.c_void_p * 1)(p.h), (C.c_void_p * 1)(img.ctypes.data), (C.c_int * 1)(img.strides[0]),
                                                    (C.c_void_p * 1)(dst.ctypes.data), (C.c_int * 1)(dst.strides[0]), 2) == M.IMP_ERROR_GPU
                assert (out == 7).all() and (dst == 7).all()
                os._exit(0)
            dev = L.init_worker(k)
            assert dev == want, (k, dev, want)
            buf = C.c_void_p()
            L.check(L.lib.imp_gpu_malloc(C.byref(buf), 1 << 20))
            assert pointer_device(buf.value) == want and current_device() == want, (pointer_device(buf.value), current_device(), want)
            L.check(L.lib.imp_gpu_free(buf))
            code, outs = api.OpsLayer(L).request([img], cfg, **rq)                # RunJob's operator calls + the flush
            assert code == 0 and np.array_equal(outs[0], ref), code
            plans = [L.plan(320, 240, 4, cfg, **rq), L.plan(130, 90, 3, cfg, **rq2)]
            dsts = [np.empty((p.out_h, p.out_w, p.out_c), np.uint8) for p in plans]
            api.run_host_batch(L, plans, [img, img2], dsts, n_streams=2)
            assert np.array_equal(dsts[0], ref) and np.array_equal(dsts[1], ref2)
            L.shutdown()
            os._exit(0)
        except BaseException as e:
            sys.stderr.write("worker %d: %r\n" % (k, e)); os._exit(1)
    pids.append(pid)
st = [os.waitpid(p, 0)[1] for p in pids]
assert all(os.WIFEXITED(s) and os.WEXITSTATUS(s) == 0 for s in st), st
print("WORKERS OK", len(pids))
""".replace("DRIVER", _CUDA_DRIVER)


def _run(code, *args):
    r = subprocess.run([sys.executable, "-c", code, *args], cwd=ROOT, capture_output=True, text=True, timeout=900,
                       env={k: v for k, v in os.environ.items() if k != "IMP_GPU_DEVICES"})
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    return r.stdout


def _devices():
    return M.library().device_count()


@pytest.mark.gpu
def test_forked_workers_take_worker_mod_n_devices():
    n = _devices()
    k = max(3, n + 1)
    assert f"WORKERS OK {k}" in _run(_WORKERS, "-", json.dumps([w % n for w in range(k)]))


@pytest.mark.gpu
def test_forked_workers_all_on_device_0():
    k = max(3, _devices() + 1)
    assert f"WORKERS OK {k}" in _run(_WORKERS, "0", json.dumps([0] * k))


@pytest.mark.gpu
def test_a_list_naming_a_missing_device_leaves_the_worker_without_one():
    n = _devices()
    assert "WORKERS OK 2" in _run(_WORKERS, str(n), json.dumps([-1, -1]))
    assert "WORKERS OK 1" in _run(_WORKERS, f"0,{n + 3}", json.dumps([-1]))


@pytest.mark.gpu
def test_forked_workers_follow_a_permuted_list():
    n = _devices()
    if n < 2:
        pytest.skip("needs two or more GPUs")
    assert "WORKERS OK 5" in _run(_WORKERS, "1,0", json.dumps([1, 0, 1, 0, 1]))
    rev = list(range(n))[::-1]
    assert f"WORKERS OK {n + 1}" in _run(_WORKERS, ",".join(map(str, rev)), json.dumps([rev[w % n] for w in range(n + 1)]))


def _farm_jobs(orc):
    cfg = dict(max_w=0, max_h=0, watermark=smooth_image(5, 12, 20, 4), wm_gravity_x="r", wm_gravity_y="b", wm_opacity=60)
    jobs = []
    for i in range(11):
        h, w, c = 60 + 17 * i, 90 + 23 * i, (3, 4)[i % 2]
        img = smooth_image(40 + i, h, w, c)
        rq = dict(crop=f"{w - 8}px,{h - 6}px,c,c", resize=f"{31 + 5 * i},{19 + 3 * i}", filters=["gamma=1.3"])
        jobs.append((img, rq, orc.run_chain(img, rq["crop"], None, rq["resize"], rq["filters"], orc.OracleConfig(**cfg))[2]))
    return cfg, jobs


@pytest.mark.gpu
def test_farm_follows_the_device_list_on_one_gpu(gpu, orc, monkeypatch):
    cfg, jobs = _farm_jobs(orc)
    plans = [gpu.plan(img.shape[1], img.shape[0], img.shape[2], api.Config(**cfg), **rq) for img, rq, _ in jobs]
    dsts = [np.full((p.out_h, p.out_w, p.out_c), 7, np.uint8) for p in plans]
    monkeypatch.setenv("IMP_GPU_DEVICES", "0")
    api.run_host_batch(gpu, plans, [j[0] for j in jobs], dsts, n_streams=2, n_gpus=1)
    for d, (_, _, ref) in zip(dsts, jobs):
        assert np.array_equal(d, ref)
    jobs_h = api.HostJobs(plans, [j[0] for j in jobs], dsts)
    for d in dsts:
        d[...] = 7
    n = gpu.device_count()
    for spec, n_gpus, code, text in [("0", 2, M.IMP_ERROR_GPU, "more GPUs requested than present"),
                                     ("0,0", 1, M.IMP_ERROR_INVALID_ARGS, 'entry 2 ("0")'),
                                     (str(n), 1, M.IMP_ERROR_INVALID_ARGS, f'entry 1 ("{n}") names no device')]:
        monkeypatch.setenv("IMP_GPU_DEVICES", spec)
        rc = gpu.lib.imp_gpu_farm_run_host(jobs_h.n, jobs_h.P, jobs_h.S, jobs_h.SS, jobs_h.D, jobs_h.DS, n_gpus, 2)
        assert rc == code and text in gpu.last_error(), (spec, rc, gpu.last_error())
        assert all((d == 7).all() for d in dsts), spec
    monkeypatch.delenv("IMP_GPU_DEVICES")
    rc = gpu.lib.imp_gpu_farm_run_host(jobs_h.n, jobs_h.P, jobs_h.S, jobs_h.SS, jobs_h.D, jobs_h.DS, n + 1, 2)
    assert rc == M.IMP_ERROR_GPU and "more GPUs requested than present" in gpu.last_error()
    for p in plans:
        p.close()


# A fresh process (no device touched yet) runs the farm under IMP_GPU_DEVICES=<argv[1]> with n_gpus = 1, 2, ...: after
# each call exactly the listed devices g < n_gpus have a context, and every result equals the oracle.
_FARM = r"""
import os, sys, numpy as np
sys.path.insert(0, "."); sys.path.insert(0, "tests")
import ngx_http_imgproc_b200 as M
from ngx_http_imgproc_b200 import api
from oracle import oracle as O
from test_worker_devices import _farm_jobs
DRIVER
spec = sys.argv[1]
os.environ["IMP_GPU_DEVICES"] = spec
lst = [int(x) for x in spec.split(",")]
L = M.library()
n = L.device_count()
cfg, jobs = _farm_jobs(O)
plans = [L.plan(img.shape[1], img.shape[0], img.shape[2], api.Config(**cfg), **rq) for img, rq, _ in jobs]
for n_gpus in range(1, len(lst) + 1):
    dsts = [np.full((p.out_h, p.out_w, p.out_c), 7, np.uint8) for p in plans]
    api.run_host_batch(L, plans, [j[0] for j in jobs], dsts, n_streams=2, n_gpus=n_gpus, policy=api.FARM_SIZE_AWARE if n_gpus % 2 else api.FARM_ROUND_ROBIN)
    for d, (_, _, ref) in zip(dsts, jobs):
        assert np.array_equal(d, ref), n_gpus
    active = [d for d in range(n) if context_active(d)]
    assert active == sorted(lst[:n_gpus]), (n_gpus, active, lst)
print("FARM OK", len(lst))
""".replace("DRIVER", _CUDA_DRIVER)


@pytest.mark.gpu
def test_farm_puts_job_shares_on_the_listed_devices():
    n = _devices()
    if n < 2:
        pytest.skip("needs two or more GPUs")
    assert "FARM OK 2" in _run(_FARM, "1,0")
    rev = ",".join(str(d) for d in range(n)[::-1])
    assert f"FARM OK {n}" in _run(_FARM, rev)


# The reference's own RunJob over the drop-in (oracle/_ref/libimp_ref_gpu.so) as nginx worker argv[1], IMP_GPU_DEVICES
# = argv[2] ("-": unset), against the CPU build's bytes; argv[3] == "bad": every request must answer IMP_ERROR_GPU.
_REF = r"""
import ctypes as C, os, sys
sys.path.insert(0, "."); sys.path.insert(0, "tests")
from oracle import oracle as O
from conftest import smooth_image
worker, spec, mode = int(sys.argv[1]), sys.argv[2], sys.argv[3]
if spec != "-": os.environ["IMP_GPU_DEVICES"] = spec
wm = smooth_image(7, 12, 20, 4)
cfgs = [O.OracleConfig(), O.OracleConfig(allow_experiments=True, max_filters=8, watermark=wm, wm_gravity_x="r", wm_gravity_y="b", wm_offset_x=3, wm_offset_y=2, wm_opacity=60)]
queries = ["crop=40,30&resize=31,17&filter-gamma=1.2&format=png", "resize=20&filter-rotate=90&filter-flip=10&format=png",
           "crop=50px,20px,c,c&filter-modulate=10,90,100&format=jpg", "resize=0,0&format=png"]
cases = []
for (h, w, c) in [(60, 80, 3), (45, 64, 4)]:
    img = smooth_image(h, h, w, c)
    for cfg in cfgs:
        for q in queries:
            cases.append((q, img, cfg, O.Ref.run_job(q, img, cfg)))
pid = os.fork()
if pid == 0:
    try:
        C.c_size_t.in_dll(C.CDLL(O.RefGpu.path()), "ngx_worker").value = worker     # the drop-in's weak ngx_worker, before OnEnvStart
        O.RefGpu.lib()                                           # OnEnvStart
        checked = 0
        for q, img, cfg, (code, step, ref) in cases:
            gcode, gstep, out = O.RefGpu.run_job(q, img, cfg)
            if mode == "bad":                                    # a request that gets as far as the flush needs the device
                assert gcode == (100 if code == 0 else code), (q, gcode, code)
                continue
            assert (gcode, gstep) == (code, step), (q, gcode, gstep, code, step)
            if code == 0:
                assert out is not None and out.shape == ref.shape and (out == ref).all(), q
                checked += 1
        assert mode == "bad" or checked >= 8, checked
        O.RefGpu.lib().OnEnvDestroy()
        os._exit(0)
    except BaseException as e:
        sys.stderr.write("worker %d: %r\n" % (worker, e)); os._exit(1)
st = os.waitpid(pid, 0)[1]
assert os.WIFEXITED(st) and os.WEXITSTATUS(st) == 0, st
print("REF OK")
"""


@pytest.mark.gpu
def test_reference_runjob_over_the_dropin_as_worker_k(orc):
    if not (orc.RefGpu.available() and orc.Ref.available()):
        pytest.skip("prebuilt oracle/_ref libraries not present on this box")
    for worker, spec, mode in [(0, "-", "ok"), (2, "-", "ok"), (2, "0", "ok"), (0, "0,,1", "bad"), (1, str(_devices()), "bad")]:
        assert "REF OK" in _run(_REF, str(worker), spec, mode)
