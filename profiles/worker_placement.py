"""What spreading nginx workers over the GPUs of a box buys: N forked workers serve cfg2 requests from pageable frames,
once all on GPU 0 (IMP_GPU_DEVICES=0) and once with the default placement (worker k on GPU k mod n).

  python profiles/worker_placement.py [--workers N] [--batch 16] [--calls 20] [--rounds 2] [--out FILE]

Each worker is a process forked from a master that loaded the library without initialising CUDA, as nginx forks its
workers; it calls imp_gpu_init_worker(k), plans cfg2 (bench.py's shapes and request), warms up, waits for the others,
then runs --calls synchronous imp_gpu_batch_run_host calls of --batch jobs over 8 distinct pageable 4K frames.
Aggregate Mpix/s = result pixels of all workers / (last worker's end - first worker's start). The two placements
alternate for --rounds rounds. The device names and power limits are read in the same run and stored with the numbers;
with one GPU both placements are the same device and the comparison says nothing.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import workload                      # noqa: E402  (the benchmark's own shapes and request)
import ngx_http_imgproc_b200 as M               # noqa: E402
from ngx_http_imgproc_b200 import api           # noqa: E402


def devices():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    return [dict(zip(("index", "name", "power_limit"), [x.strip() for x in line.split(",")])) for line in q.strip().splitlines()]


def worker(L, k, batch, calls, go_r, out_w):
    wl = workload("cfg2")
    (shape, rq, _), = wl["jobs"]
    h, w, c = shape
    dev = L.init_worker(k)
    plan = L.plan(w, h, c, api.Config(**wl["cfg"]), **rq)
    rng = np.random.default_rng(100 + k)
    frames = [rng.integers(0, 256, shape, dtype=np.uint8) for _ in range(8)]
    outs = [np.empty((plan.out_h, plan.out_w, plan.out_c), np.uint8) for _ in range(batch)]
    jobs = api.HostJobs([plan] * batch, [frames[i % len(frames)] for i in range(batch)], outs)
    jobs.run(L, n_streams=4)                                   # warm-up: plan upload, lanes, staging, copy workers
    os.write(out_w, b"ready\n")
    os.read(go_r, 1)
    t0 = time.perf_counter()                                   # CLOCK_MONOTONIC: comparable across the workers
    for _ in range(calls):
        jobs.run(L, n_streams=4)
    t1 = time.perf_counter()
    os.write(out_w, (json.dumps({"worker": k, "device": dev, "t0": t0, "t1": t1, "pixels": calls * batch * plan.out_w * plan.out_h}) + "\n").encode())
    L.shutdown()


def run_placement(L, spec, n_workers, batch, calls):
    if spec is None:
        os.environ.pop("IMP_GPU_DEVICES", None)
    else:
        os.environ["IMP_GPU_DEVICES"] = spec
    go_r, go_w = os.pipe()
    out_r, out_w = os.pipe()
    pids = []
    for k in range(n_workers):
        pid = os.fork()
        if pid == 0:
            code = 0
            try:
                worker(L, k, batch, calls, go_r, out_w)
            except BaseException as e:
                sys.stderr.write("worker %d: %r\n" % (k, e))
                code = 1
            os._exit(code)
        pids.append(pid)
    f = os.fdopen(out_r)
    for _ in range(n_workers):
        assert f.readline().strip() == "ready"
    os.write(go_w, b"g" * n_workers)
    res = [json.loads(f.readline()) for _ in range(n_workers)]
    st = [os.waitpid(p, 0)[1] for p in pids]
    assert all(os.WIFEXITED(s) and os.WEXITSTATUS(s) == 0 for s in st), st
    f.close(); os.close(go_r); os.close(go_w); os.close(out_w)
    span = max(r["t1"] for r in res) - min(r["t0"] for r in res)
    return {"IMP_GPU_DEVICES": spec, "devices": sorted(r["device"] for r in res), "seconds": span,
            "aggregate_mpix_s": sum(r["pixels"] for r in res) / span / 1e6,
            "per_worker_mpix_s": [r["pixels"] / (r["t1"] - r["t0"]) / 1e6 for r in sorted(res, key=lambda r: r["worker"])]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workers", type=int, default=0, help="default: one per GPU")
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    gpus = devices()                                           # nvidia-smi: this process itself stays without CUDA
    if not gpus:
        raise SystemExit("no GPU: nothing to measure")
    n_workers = a.workers or len(gpus)
    L = M.library()
    res = {"what": __doc__.strip().splitlines()[0], "gpus": gpus, "workers": n_workers, "batch": a.batch, "calls": a.calls,
           "request": "cfg2 (bench.py), pageable frames", "runs": []}
    for _ in range(a.rounds):
        for spec in ("0", None):
            r = run_placement(L, spec, n_workers, a.batch, a.calls)
            res["runs"].append(r)
            print(json.dumps({k: r[k] for k in ("IMP_GPU_DEVICES", "devices", "aggregate_mpix_s")}), flush=True)
    med = lambda spec: float(np.median([r["aggregate_mpix_s"] for r in res["runs"] if r["IMP_GPU_DEVICES"] == spec]))
    res["shared_gpu0_mpix_s"], res["default_mpix_s"] = med("0"), med(None)
    res["default_over_shared"] = res["default_mpix_s"] / res["shared_gpu0_mpix_s"]
    if len(gpus) < 2:
        res["note"] = "one GPU: both placements use device 0, the ratio is noise"
    print(json.dumps({k: res[k] for k in ("workers", "shared_gpu0_mpix_s", "default_mpix_s", "default_over_shared")}))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
