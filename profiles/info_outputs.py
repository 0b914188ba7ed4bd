"""What a format=json / format=text request saves by bringing back the answer instead of the frame.

  python profiles/info_outputs.py [--calls 10] [--out profiles/r03_info_outputs.json]

Batch legs: cfg1, cfg2 and cfg4 of bench.py through the host-batch path with pinned and with pageable sources (32 distinct
seeded frames per shape, cycled), three ways: FRAME (imp_gpu_batch_run_host, results into pinned / pageable frames),
BRIGHTNESS (imp_gpu_batch_brightness_host) and ASCII (imp_gpu_batch_ascii_host, every other job with the wide ramp). Each
leg: every shape warmed up first, then the median, best and worst of --calls synchronous calls.
One request: what Info() costs today after the operator layer (imp_FlushAll, then the reference's column-major float loop
over the host result, orc.perceived_brightness) against imp_Brightness on the recorded frame; pageable frames, as
cvDecodeImage hands them over.
Bytes: device-to-host bytes per job, from the shapes.
The device name and power limit are read in the same run and stored with the numbers.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import workload                      # noqa: E402  (the benchmark's own shapes and requests)
import ngx_http_imgproc_b200 as M               # noqa: E402
from ngx_http_imgproc_b200 import api           # noqa: E402

CONFIGS = ("cfg1", "cfg2", "cfg4")


def timed(fn, calls):
    fn()                                                               # warm-up: plans uploaded, lanes and staging sized
    t = []
    for _ in range(calls):
        t0 = time.perf_counter(); fn(); t.append(time.perf_counter() - t0)
    return {"median_ms": statistics.median(t) * 1e3, "best_ms": min(t) * 1e3, "worst_ms": max(t) * 1e3, "calls": calls}


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    name, power, clock = ([x.strip() for x in q.split(",")] + ["?", "?", "?"])[:3]
    return {"name": name, "power_limit": power, "sm_max_clock": clock}


def batch_legs(L, name, calls):
    import torch
    wl = workload(name)
    (shape, rq, n), = wl["jobs"]
    h, w, c = shape
    plan = L.plan(w, h, c, api.Config(**wl["cfg"]), **rq)
    rng = np.random.default_rng(5)
    pool = [rng.integers(0, 256, shape, dtype=np.uint8) for _ in range(min(32, n))]
    pinned = [torch.from_numpy(a).pin_memory() for a in pool]
    out_shape = (plan.out_h, plan.out_w, plan.out_c)
    text_len = L.lib.imp_gpu_ascii_length(plan.out_w, plan.out_h)
    plans = [plan] * n
    res = {"jobs": n, "request": rq, "source": list(shape), "result": list(out_shape),
           "d2h_bytes_per_job": {"frame": int(np.prod(out_shape)), "brightness": 4, "ascii": int(text_len)}}
    for kind in ("pinned", "pageable"):
        srcs = [(pinned[k % len(pool)].numpy() if kind == "pinned" else pool[k % len(pool)]) for k in range(n)]
        if kind == "pinned":
            douts = [torch.empty(out_shape, dtype=torch.uint8).pin_memory() for _ in range(min(32, n))]
            dsts = [douts[k % len(douts)].numpy() for k in range(n)]
        else:
            douts = [np.empty(out_shape, np.uint8) for _ in range(min(32, n))]
            dsts = [douts[k % len(douts)] for k in range(n)]
        frames = api.HostJobs(plans, srcs, dsts)
        P, S, SS = api._job_arrays(plans, srcs)
        bright = np.zeros(n, np.float32)
        texts = [C.create_string_buffer(text_len) for _ in range(n)]
        T = (C.c_void_p * n)(*[C.addressof(t) for t in texts])
        caps = (C.c_long * n)(*([text_len] * n))
        A = (C.c_char_p * n)(*[b"wide" if k % 2 else None for k in range(n)])
        res[kind] = {
            "frame": timed(lambda: frames.run(L, n_streams=4), calls),
            "brightness": timed(lambda: L.check(L.lib.imp_gpu_batch_brightness_host(n, P, S, SS, bright.ctypes.data, 4)), calls),
            "ascii": timed(lambda: L.check(L.lib.imp_gpu_batch_ascii_host(n, P, S, SS, A, T, caps, 4)), calls),
        }
        del frames, douts
    plan.close()
    return res


def one_request(L, name, calls):
    from oracle import oracle as O
    o = O.orc()
    wl = workload(name)
    (shape, rq, _), = wl["jobs"]
    cfg = api.Config(**wl["cfg"])
    img = np.random.default_rng(6).integers(0, 256, shape, dtype=np.uint8)
    ops = api.OpsLayer(L)
    req = dict(crop=rq.get("crop"), resize=rq.get("resize"), filters=rq.get("filters", ()))

    def today():
        code, outs = ops.request([img], cfg, **req)
        assert code == 0
        return o.perceived_brightness(outs[0])

    def answer():
        code, b = ops.brightness([img], cfg, **req)
        assert code == 0
        return b[0]

    a, b = today(), answer()
    return {"flushall_then_host_loop": timed(today, calls), "imp_Brightness": timed(answer, calls),
            "values": {"host_loop": a, "imp_Brightness": b}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_info_outputs.json"))
    a = ap.parse_args()
    L = M.library()
    L.init(0)
    res = {"device": device_info(), "what": __doc__.strip().splitlines()[0], "batch": {}, "one_request": {}}
    for name in CONFIGS:
        res["batch"][name] = batch_legs(L, name, max(10, a.calls))
        res["one_request"][name] = one_request(L, name, max(10, a.calls))
        print(name, json.dumps({k: {leg: round(v[leg]["median_ms"], 3) for leg in ("frame", "brightness", "ascii")} for k, v in res["batch"][name].items()
                                if k in ("pinned", "pageable")}), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
