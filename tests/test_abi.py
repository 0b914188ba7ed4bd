"""CPU tests of the drop-in boundary: libimp_gpu.so builds, loads, exports every symbol the headers
declare, validates requests without a GPU, and refuses to compute without one (no CPU fallback)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import ngx_http_imgproc_b200 as M
from conftest import ROOT


def _declared(header):
    text = open(os.path.join(ROOT, "include", header)).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(imp_gpu_[a-z0-9_]+|imp_ops_[a-z0-9_]+|imp_(?:Crop|Resize|Watermark|Filter|BlendWithPaper|Flush|[A-Z][A-Za-z0-9]+))\s*\(", text)))


def test_library_builds_and_exports_every_declared_symbol():
    path = M.build()
    assert os.path.exists(path)
    lib = C.CDLL(path)
    headers = [h for h in os.listdir(os.path.join(ROOT, "include")) if h.endswith(".h")]
    assert "imp_gpu.h" in headers
    total = 0
    for h in headers:
        for sym in _declared(h):
            assert hasattr(lib, sym), f"{h} declares {sym} but libimp_gpu.so does not export it"
            total += 1
    assert total >= 30


def test_only_sm100a_code_in_the_library():
    import shutil, subprocess
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "-lelf", M.build()], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_validation_needs_no_gpu_and_matches_reference_codes():
    L = M.library()
    code, step, plan = L.try_plan(1920, 1080, 3, resize="640,360")
    assert code == 0 and (plan.out_w, plan.out_h, plan.out_c) == (640, 360, 3)
    assert plan.algorithmic_bytes == 1920 * 1080 * 3 + 640 * 360 * 3           # SURVEY §8d cfg1: 6.912 MB
    plan.close()
    assert L.try_plan(100, 100, 3, crop="400px,200")[:2] == (50, 3)
    assert L.try_plan(100, 100, 3, resize="3000,0,up")[:2] == (54, 4)
    assert L.try_plan(100, 100, 3, filters=["vignette=0.8"])[:2] == (52, 5)
    assert L.try_plan(100, 100, 3, filters=["gamma=1"] * 6)[:2] == (55, 0)
    code, step, plan = L.try_plan(3840, 2160, 4, M.Config(watermark=np.zeros((64, 256, 4), np.uint8), wm_gravity_x="r", wm_gravity_y="b",
                                                         wm_offset_x=10, wm_offset_y=10, wm_opacity=60), crop="3600px,2025px,c,c", resize="800,450")
    assert code == 0 and plan.window == (120, 68, 3600, 2025) and (plan.out_w, plan.out_h) == (800, 450)
    assert plan.algorithmic_bytes == 29160000 + 1440000 + 65536                # SURVEY §8d cfg2: 30.67 MB
    plan.close()


def test_farm_rejects_a_negative_job_count():
    """A negative n is an argument error (with or without a device), never an exception escaping the C ABI."""
    L = M.library()
    for fn in (L.lib.imp_gpu_farm_run_host_policy, L.lib.imp_gpu_farm_run_host):
        extra = (1, 4, 0) if fn is L.lib.imp_gpu_farm_run_host_policy else (1, 4)
        assert fn(-1, None, None, None, None, None, *extra) == M.IMP_ERROR_INVALID_ARGS


def test_no_cpu_fallback_without_a_gpu():
    """On a box without a GPU every compute entry point must fail with IMP_ERROR_GPU, never produce pixels."""
    L = M.library()
    if L.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(M.ImpError) as e:
        L.init(0)
    assert e.value.code == M.IMP_ERROR_GPU
    plan = L.plan(8, 8, 3, resize="4,4")
    out = np.full((4, 4, 3), 7, np.uint8)
    with pytest.raises(M.ImpError) as e:
        plan.run_host(np.zeros((8, 8, 3), np.uint8), out)
    assert e.value.code == M.IMP_ERROR_GPU and (out == 7).all()
    plan.close()


def test_product_does_not_reference_the_oracle():
    """Nothing under ngx_http_imgproc_b200/ or include/ may import, link or name oracle/."""
    bad = []
    for base in ("ngx_http_imgproc_b200", "include"):
        for dp, _, files in os.walk(os.path.join(ROOT, base)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h", ".c")):
                    if re.search(r"\boracle\b|imp_oracle|hostsim", open(os.path.join(dp, f), errors="ignore").read()):
                        bad.append(os.path.join(dp, f))
    assert not bad, bad


def test_headers_are_plain_c_and_a_c_host_links(tmp_path):
    """The boundary is a C ABI for a C host (bridge.c): both public headers compile as strict C99 and a C program links against
    libimp_gpu.so, validates a request (no GPU needed) and sees IMP_ERROR_GPU — never a fallback — from a compute call."""
    import subprocess
    src = tmp_path / "host.c"
    src.write_text(r'''
#include <stdio.h>
#include <string.h>
#include "imp_gpu.h"
#include "imp_ops.h"
int main(void) {
    imp_gpu_request rq; imp_gpu_config cfg; imp_gpu_plan* plan = NULL; int step = -1, w, h, c, rc;
    const char* filters[2] = {"gamma=1.2", "rotate=90"};
    int owner[3]; imp_gpu_plan* plans[3];
    memset(&rq, 0, sizeof rq); memset(&cfg, 0, sizeof cfg);
    cfg.max_filters = 5;
    rq.crop = "400px,300px,c,c"; rq.resize = "200"; rq.filters = filters; rq.filter_count = 2;
    rc = imp_gpu_plan_create(&rq, &cfg, 640, 480, 3, &plan, &step);
    if (rc != IMP_OK) return 1;
    imp_gpu_plan_output(plan, &w, &h, &c);
    if (w != 150 || h != 200 || c != 3 || imp_gpu_plan_passes(plan) != 1) return 2;      /* 200x150 rotated */
    plans[0] = plans[1] = plans[2] = plan;
    if (imp_gpu_farm_assign(3, plans, 2, IMP_FARM_SIZE_AWARE, owner) != IMP_OK || owner[0] == owner[1]) return 3;
    rq.resize = "0,0";
    { imp_gpu_plan* bad = NULL; if (imp_gpu_plan_create(&rq, &cfg, 640, 480, 3, &bad, &step) != IMP_ERROR_INVALID_ARGS || step != IMP_STEP_RESIZE) return 4; }
    if (imp_gpu_device_count() == 0) {
        unsigned char px[640 * 480 * 3], out[150 * 200 * 3];
        memset(px, 7, sizeof px);
        if (imp_gpu_init(0) != IMP_ERROR_GPU) return 5;
        if (imp_gpu_run_host(plan, px, 640 * 3, out, 150 * 3) != IMP_ERROR_GPU) return 6;    /* no CPU fallback */
        if (strlen(imp_gpu_last_error()) == 0) return 7;
    }
    imp_gpu_plan_destroy(plan);
    printf("C HOST OK %d\n", (int)sizeof(IplImage));
    return 0;
}
''')
    exe = tmp_path / "host"
    pkg = os.path.join(ROOT, "ngx_http_imgproc_b200")
    r = subprocess.run(["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src),
                        "-L", pkg, "-limp_gpu", "-Wl,-rpath," + pkg], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0 and "C HOST OK 144" in r.stdout, (r.returncode, r.stdout, r.stderr)
