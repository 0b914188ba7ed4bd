"""Brightness and ASCII answers (imp_gpu_batch_brightness_host, imp_gpu_batch_ascii_host, imp_Brightness, imp_Ascii) have no
CPU path: without a device every one of them returns IMP_ERROR_GPU and leaves its outputs as they were."""
import ctypes as C

import numpy as np
import pytest

import ngx_http_imgproc_b200 as M
from ngx_http_imgproc_b200 import api
from conftest import rnd_image


@pytest.fixture
def no_gpu_lib():
    L = M.library()
    if L.device_count() > 0:
        pytest.skip("a GPU is present")
    return L


def test_batch_answers_fail_without_a_gpu_and_write_nothing(no_gpu_lib):
    L = no_gpu_lib
    imgs = [rnd_image(1, 24, 40, 3), rnd_image(2, 17, 9, 4)]
    plans = [L.plan(40, 24, 3, resize="20,12"), L.plan(9, 17, 4)]
    P = (C.c_void_p * 2)(*[p.h for p in plans])
    S = (C.c_void_p * 2)(*[i.ctypes.data for i in imgs])
    SS = (C.c_int * 2)(*[i.strides[0] for i in imgs])
    b = np.full(2, -7.0, np.float32)
    assert L.lib.imp_gpu_batch_brightness_host(2, P, S, SS, b.ctypes.data, 4) == M.IMP_ERROR_GPU
    assert (b == -7.0).all()
    lens = [L.lib.imp_gpu_ascii_length(p.out_w, p.out_h) for p in plans]
    bufs = [C.create_string_buffer(b"\x5a" * k, k) for k in lens]
    T = (C.c_void_p * 2)(*[C.addressof(x) for x in bufs])
    A = (C.c_char_p * 2)(b"wide", None)
    caps = (C.c_long * 2)(*lens)
    assert L.lib.imp_gpu_batch_ascii_host(2, P, S, SS, A, T, caps, 4) == M.IMP_ERROR_GPU
    assert all(x.raw == b"\x5a" * k for x, k in zip(bufs, lens))
    assert L.last_error()
    with pytest.raises(M.ImpError) as e:
        L.batch_brightness(plans, imgs)
    assert e.value.code == M.IMP_ERROR_GPU
    for p in plans:
        p.close()


def test_answer_operators_fail_without_a_gpu_and_keep_the_recording(no_gpu_lib):
    L = no_gpu_lib
    ops = api.OpsLayer(L)
    img = rnd_image(3, 30, 50, 3)
    code, ptrs = ops.record([img], api.Config(), resize="25,15", filters=["rotate=90"])
    assert code == 0
    p = ptrs[0]
    assert L.lib.imp_ops_pending(p) == 2
    v = C.c_float(-7.0)
    assert L.lib.imp_Brightness(p, C.byref(v)) == M.IMP_ERROR_GPU and v.value == -7.0
    n = L.lib.imp_gpu_ascii_length(p.contents.width, p.contents.height)
    buf = C.create_string_buffer(b"\x5a" * n, n)
    assert L.lib.imp_Ascii(p, b"wide", buf, n) == M.IMP_ERROR_GPU and buf.raw == b"\x5a" * n
    assert L.lib.imp_ops_pending(p) == 2 and (p.contents.width, p.contents.height) == (15, 25)
    L.lib.imp_Discard(p)
