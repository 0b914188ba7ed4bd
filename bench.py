#!/usr/bin/env python
"""
bench.py — output Mpix/s of IMP's fused decoded-pixel chain on B200 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config cfg2] [--impl ours|reference] [--extras all|none|cfg1,cfg5]
                  [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic frames. The headline workload is BASELINE.json
configs[1] (cfg2): 256 requests of a 3840x2160 BGRA frame -> crop 3600x2025 -> INTER_AREA to 800x450 -> 256x64 watermark
at opacity 60, i.e. one fused kernel launch over 256 jobs.

  value        whole-job Mpix/s with the frames already resident in HBM (CUDA events, max over ranks)
  e2e          the same metric through the public C ABI with HOST (pinned) buffers: H2D of every request's crop window +
               kernels + D2H of every result inside the timed region (median of >= 10 steps; min and max beside it)
  roofline     algorithmic bytes (SURVEY §8d) / measured launch time / MEASURED_PEAKS.json hbm_gbs
  cpu_baseline the reference's CPU path (its own C for filters/compositing compiled unmodified + cv2 for the OpenCV
               calls; or the C port when those are absent) on this box's host cores: all cores as independent
               single-threaded worker processes (how nginx scales) AND one worker alone
  extra_configs  the other BASELINE configs (cfg1, cfg3, cfg3nn, cfg4, cfg5) measured the same way in the same run:
               {ms_per_step, value, roofline, e2e, cpu_baseline} each (N=1: all; N>1: cfg5 strong-scaled)
  request_latency_ms  one request at a time: imp_gpu_run_host on a warm plan, and the whole operator sequence of RunJob
               (imp_Crop .. imp_FlushAll) for a repeated request and with the plan cache emptied first (cold: planner + upload)
  h2d_ceiling  bare concurrent pinned cudaMemcpyAsync H2D on all ranks: the box's ceiling for the e2e numbers

Multi-GPU: one process per GPU (torchrun). The headline is weak-scaled (every rank runs the cfg2 batch on its own frames;
frames are independent, there is no collective on the data path). cfg5 (BASELINE configs[4], "sharded across 2/4/8 B200")
is STRONG-scaled in extra_configs: the same 65,536 jobs, job i on GPU i mod N (and a size-aware assignment), plus one
imp_gpu_farm_run_host call from rank 0 over all N GPUs. `--impl reference` times the reference CPU implementation only
(rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "output Mpix/s (fused resize+filter chain)"
EXTRA_ORDER = ["cfg1", "cfg3", "cfg3nn", "cfg4", "cfg5"]


# ------------------------------------------------------------------------------------------------------------
# Workloads (SURVEY §8d). Each: list of (src_shape(h,w,c), request kwargs, n_jobs_with_this_shape), cfg kwargs
# ------------------------------------------------------------------------------------------------------------
def watermark(seed, h, w):
    rng = np.random.default_rng(seed)
    wm = rng.integers(0, 256, (h, w, 4), dtype=np.uint8)
    wm[:, :, 3] = np.linspace(0, 255, w).astype(np.uint8)[None, :]
    return wm


def workload(name: str, scale: int = 1):
    if name == "cfg1":
        return dict(desc="1920x1080x3 -> resize=640,360 (AREA 3x3), batch 256", jobs=[((1080, 1920, 3), dict(resize="640,360"), 256 // scale)], cfg=dict())
    if name == "cfg1l":   # cfg1 "as worded": bilinear (shim-level extension, not a reference call site)
        return dict(desc="1920x1080x3 -> resize=640,360 INTER_LINEAR (extension), batch 256", jobs=[((1080, 1920, 3), dict(resize="640,360", interp=1), 256 // scale)], cfg=dict())
    if name == "cfg3nn":  # cfg3 reference-faithful: GIF output forces INTER_NN (bridge.c:594)
        return dict(desc="200 frames 480x270x4 -> resize=960,540,up (NN, GIF output) + modulate=0,0,100 + colorize=704214,0.6",
                    jobs=[((270, 480, 4), dict(resize="960,540,up", simple=True, filters=["modulate=0,0,100", "colorize=704214,0.6"]), 200 // scale)], cfg=dict())
    if name == "cfg2":
        return dict(desc="256 x [3840x2160x4 -> crop=3600px,2025px,c,c -> resize=800,450 (AREA 4.5x) -> 256x64 watermark r,b,10,10 opacity 60]",
                    jobs=[((2160, 3840, 4), dict(crop="3600px,2025px,c,c", resize="800,450"), 256 // scale)],
                    cfg=dict(watermark=watermark(3, 64, 256), wm_gravity_x="r", wm_gravity_y="b", wm_offset_x=10, wm_offset_y=10, wm_opacity=60))
    if name == "cfg3":
        return dict(desc="200 frames 480x270x4 -> resize=960,540,up (CUBIC 2x) + modulate=0,0,100 + colorize=704214,0.6",
                    jobs=[((270, 480, 4), dict(resize="960,540,up", filters=["modulate=0,0,100", "colorize=704214,0.6"]), 200 // scale)], cfg=dict())
    if name == "cfg4":
        return dict(desc="8 x [4000x3000x3 -> blur=2.3 + vignette=0.8 + rotate=90]",
                    jobs=[((3000, 4000, 3), dict(filters=["blur=2.3", "vignette=0.8", "rotate=90"]), max(1, 8 // scale))], cfg=dict(allow_experiments=True))
    if name == "cfg5":
        rng = np.random.default_rng(6)
        shapes = [(int(rng.integers(240, 1537)), int(rng.integers(320, 2049)), 3 if rng.random() < 0.75 else 4) for _ in range(512)]
        n = 65536 // scale
        per = [n // 512 + (1 if i < n % 512 else 0) for i in range(512)]
        return dict(desc=f"{n} jobs over 512 mixed-size sources (job j reads source j mod 512) -> resize=256,256 (AREA) + 64x64 watermark r,b,8,8",
                    jobs=[(s, dict(resize="256,256"), k) for s, k in zip(shapes, per) if k], interleave=True,
                    cfg=dict(max_w=0, max_h=0, watermark=watermark(61, 64, 64), wm_gravity_x="r", wm_gravity_y="b", wm_offset_x=8, wm_offset_y=8, wm_opacity=100))
    raise SystemExit(f"unknown config {name}")


def job_order(wl):
    """Shape index of every job, in submission order. cfg5: job j uses source j mod 512 (consecutive jobs, hence
    consecutive CTAs, never share a frame: the 1.7 GB pool is cycled and nothing is served from the 126 MB L2)."""
    counts = [k for _, _, k in wl["jobs"]]
    if not wl.get("interleave"):
        return [i for i, k in enumerate(counts) for _ in range(k)]
    order, left = [], list(counts)
    while any(left):
        for i in range(len(left)):
            if left[i]:
                order.append(i); left[i] -= 1
    return order


# ------------------------------------------------------------------------------------------------------------
# CPU reference arm
# ------------------------------------------------------------------------------------------------------------
def _cpu_worker(args):
    """One nginx-worker-like process: runs `count` requests of the workload single-threaded."""
    name, scale, count, seed, use_ref = args
    from oracle import oracle as O
    wl = workload(name, scale)
    cfg = O.OracleConfig(**wl["cfg"])
    rng = np.random.default_rng(seed)
    shapes = wl["jobs"]
    picks = [shapes[(seed + 7 * k) % len(shapes)] for k in range(min(count, 8))]        # mixed-size farm: a spread of its shapes
    imgs = [rng.integers(0, 256, s[0], dtype=np.uint8) for s in picks]
    ref_ok = False
    if use_ref and O.Ref.available():
        ref_ok = O.Ref.use_cv2(True)
    # output pixels per request, from the port, outside the timed region (a GIF-encoded answer is not decoded back)
    pix = []
    for (shape, rq, _), img in zip(picks, imgs):
        code, step, out = O.run_chain(img, rq.get("crop"), None, rq.get("resize"), rq.get("filters", []), cfg, bool(rq.get("simple")))
        assert code == 0
        pix.append(out.shape[0] * out.shape[1])
    t0 = time.perf_counter()
    opix = 0
    for k in range(count):
        shape, rq, _ = picks[k % len(picks)]
        img = imgs[k % len(picks)]
        if ref_ok:
            query = "&".join(([f"crop={rq['crop']}"] if rq.get("crop") else []) + ([f"resize={rq['resize']}"] if rq.get("resize") else []) +
                             [f"filter-{f}" for f in rq.get("filters", [])])
            if rq.get("simple"):
                query += "&format=gif"
            code, step, out = O.Ref.run_job(query, img, cfg)
        else:
            code, step, out = O.run_chain(img, rq.get("crop"), None, rq.get("resize"), rq.get("filters", []), cfg, bool(rq.get("simple")))
        assert code == 0
        opix += pix[k % len(picks)]
    return time.perf_counter() - t0, opix, ref_ok


def cpu_run(name, scale, per_worker, workers, use_ref=True):
    """`workers` independent single-threaded processes (how nginx worker_processes scales). Returns Mpix/s, kind, wall."""
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    with ctx.Pool(workers) as pool:
        res = pool.map(_cpu_worker, [(name, scale, per_worker, 1000 + i, use_ref) for i in range(workers)])
    wall = max(r[0] for r in res)
    opix = sum(r[1] for r in res)
    kind = "reference" if all(r[2] for r in res) else "port"
    return opix / wall / 1e6, kind, wall


CPU_PER_WORKER = {"cfg2": 12, "cfg4": 1, "cfg1": 60, "cfg1l": 60, "cfg3": 40, "cfg3nn": 150, "cfg5": 24}


def cpu_baseline(name, scale, cores):
    """SURVEY §8d CPU baseline: (ii) all cores as single-threaded workers, and (i) one worker alone."""
    per = CPU_PER_WORKER.get(name, 8)
    try:
        v, kind, wall = cpu_run(name, scale, per, cores)
        v1, kind1, wall1 = cpu_run(name, scale, max(1, per // 2), 1)
        return {"value": v, "unit": "Mpix/s", "cores": cores, "kind": kind,
                "sample": f"{per} request(s) x {cores} single-threaded worker processes ({wall:.1f} s), same request as '{name}'",
                "single_worker": {"value": v1, "unit": "Mpix/s", "cores": 1, "sample": f"{max(1, per // 2)} request(s), one process ({wall1:.1f} s)"}}
    except Exception as ex:  # the baseline must not take the GPU numbers down with it
        return {"value": None, "unit": "Mpix/s", "cores": cores, "kind": "port", "sample": f"failed: {ex}"}


# ------------------------------------------------------------------------------------------------------------
def sample_clocks(stop, out):
    q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    idx = os.environ.get("LOCAL_RANK", "0")
    while not stop.is_set():
        try:
            r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", idx], capture_output=True, text=True, timeout=5)
            f = [x.strip() for x in r.stdout.strip().split(",")]
            if len(f) >= 6:
                out.append(f)
        except Exception:
            pass
        stop.wait(0.15)


def clocks_summary(samples):
    if not samples:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
    sm = [float(s[0]) for s in samples if s[0].replace(".", "").isdigit()]
    mx = [float(s[1]) for s in samples if s[1].replace(".", "").isdigit()]
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in samples)]
    return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(samples)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def _bind_to_gpu_cpus(index: int) -> bool:
    """Multi-GPU runs: pin this rank to the CPUs NVML reports as local to its GPU before any pinned host memory is
    allocated, so the e2e leg's staging buffers are first-touched on the GPU's own NUMA node (the H2D copies of 8 ranks
    otherwise cross the socket interconnect). Best effort: silently skipped where NVML or the cpuset says no."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {i * 64 + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return False
        os.sched_setaffinity(0, cpus)
        return True
    except Exception:
        return False


def config_dict(name, wl, **more):
    """The `config` object both arms print (identical by construction: it depends on the workload alone)."""
    l2 = ("512 sources (1.7 GB) cycled job by job (job j reads source j mod 512): consecutive CTAs never share a frame" if wl.get("interleave")
          else "every job has its own source frame; inputs per step >> 126 MB L2 (no flush needed)")
    d = {"workload": name + ": " + wl["desc"], "l2": l2}
    d.update(more)
    return d


class Ctx:
    """What every measurement needs: the library, torch, this rank's place in the job."""

    def __init__(self, a):
        import torch
        import ngx_http_imgproc_b200 as M
        from ngx_http_imgproc_b200 import api
        self.torch, self.api, self.a = torch, api, a
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.numa_bound = _bind_to_gpu_cpus(self.local) if self.world > 1 else False
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist
            # a CPU-side group: ranks that must WAIT while rank 0 drives their GPU from its own process (the farm leg) may
            # not sit in an NCCL barrier, whose kernel spins on the GPU and time-slices with rank 0's context
            self.cpu_group = dist.new_group(backend="gloo")
        self.L = M.library()
        self.L.init(self.local)
        self.dev = torch.device("cuda", self.local)
        self.tstream = torch.cuda.Stream(device=self.dev)      # a real (non-default) stream: kernels and the events that time them
        self.peak, self.peak_src = peaks()

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def cpu_barrier(self):
        self.torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier(group=self.cpu_group)

    def allmax(self, v: float) -> float:
        if self.dist is None:
            return float(v)
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(self, v: float) -> float:
        if self.dist is None:
            return float(v)
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())


def lpt_assign(costs, n):
    """Largest job first onto the least-loaded GPU (the size-aware sharding of SURVEY §8e); returns owner per job."""
    import heapq
    heap = [(0, g) for g in range(n)]
    owner = [0] * len(costs)
    for i in sorted(range(len(costs)), key=lambda i: -costs[i]):
        load, g = heapq.heappop(heap)
        owner[i] = g
        heapq.heappush(heap, (load + costs[i], g))
    return owner


DUMP_BYTES = 60 << 20          # --dump-outputs: float32 pixels written in all, under 64 MB with the .npy headers


def dump_sample(n_jobs: int, job_shape, budget: int = DUMP_BYTES):
    """The frames --dump-outputs writes: [(job, rows)] in submission order. Jobs are taken in a fixed seeded permutation while
    their float32 frames fit the budget; rows is None for a whole frame. When the first job's frame alone is over the budget,
    it is the only one, cut to a fixed seeded sample of its rows (sorted). The same workload always gives the same sample."""
    rng = np.random.default_rng(2024)
    pick, total = [], 0
    for j in rng.permutation(n_jobs).tolist():
        h, w, c = job_shape(j)
        if total + 4 * h * w * c <= budget:
            pick.append((j, None)); total += 4 * h * w * c
            continue
        if not pick:
            pick.append((j, np.sort(rng.choice(h, max(1, budget // (4 * w * c)), replace=False))))
        break
    return sorted(pick, key=lambda p: p[0])


def write_dump(path: str, name: str, frames) -> None:
    """frames: [(job index, HxWxC uint8 array)] -> <path>/<name>_job<index>.npy as float32 (exact for bytes)."""
    os.makedirs(path, exist_ok=True)
    for j, f in frames:
        np.save(os.path.join(path, f"{name}_job{j:05d}.npy"), f.astype(np.float32))


def measure(cx: Ctx, name: str, steps: int, warmup: int, e2e_steps: int, shard: str = "weak", seed_off: int = 0, dump: bool = False):
    """Device-resident batch (CUDA events) + end-to-end host batch of one workload on this rank.
    shard: "weak" = every rank runs the whole workload on its own frames; "mod" / "lpt" = the workload's jobs are split
    over the ranks (strong scaling): job i on GPU i mod N, or largest-first by algorithmic bytes.
    dump: keep a sample of the frames the last timed step wrote (res["_dump"], see dump_sample) for --dump-outputs."""
    torch, api, L, dev = cx.torch, cx.api, cx.L, cx.dev
    wl = workload(name, cx.a.scale)
    cfg = api.Config(**wl["cfg"])
    gen = torch.Generator(device=dev); gen.manual_seed(1234 + cx.rank + seed_off)
    order = job_order(wl)
    plans = [L.plan(s[1], s[0], s[2], cfg, **rq) for s, rq, _ in wl["jobs"]]
    if shard == "weak":
        mine = list(range(len(order)))
    elif shard == "mod":
        mine = [j for j in range(len(order)) if j % cx.world == cx.rank]
    else:
        owner = lpt_assign([plans[order[j]].algorithmic_bytes for j in range(len(order))], cx.world)
        mine = [j for j in range(len(order)) if owner[j] == cx.rank]
    # device-resident frames: one source per job (cfg5: the 512-source pool, cycled) and one destination per job
    per_shape = {}
    for j in mine:
        per_shape[order[j]] = per_shape.get(order[j], 0) + 1
    srcs, dsts = {}, {}
    for si, cnt in per_shape.items():
        (h, w, c), _, _ = wl["jobs"][si]
        p = plans[si]
        pitch = (w * c + 15) & ~15
        n_src = cnt if not wl.get("interleave") else 1
        srcs[si] = torch.randint(0, 256, (n_src, h, pitch), dtype=torch.uint8, device=dev, generator=gen)
        opitch = (p.out_w * p.out_c + 15) & ~15
        dsts[si] = torch.empty((cnt, p.out_h, opitch), dtype=torch.uint8, device=dev)
    batch = api.Batch(L)
    used = {si: 0 for si in per_shape}
    out_pix = 0
    slots = []
    for j in mine:
        si = order[j]
        p = plans[si]
        k = used[si]; used[si] += 1
        s = srcs[si]
        batch.add(p, s[k % s.shape[0]].data_ptr(), s.shape[2], dsts[si][k].data_ptr(), dsts[si].shape[2])
        slots.append((j, si, k))
        out_pix += p.out_w * p.out_h
    torch.cuda.synchronize()
    torch.cuda.set_stream(cx.tstream)
    stream = cx.tstream.cuda_stream
    assert stream != 0
    batch.launch(stream)                      # compiles the job table
    torch.cuda.synchronize()
    algo_bytes = batch.algorithmic_bytes
    for _ in range(max(warmup, 3)):
        batch.launch(stream)
    cx.barrier()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    l0 = L.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s, e in evs:
        s.record(); batch.launch(stream); e.record()
    e1.record()
    cx.barrier()
    launches = L.launch_count() - l0
    total_ms = cx.allmax(e0.elapsed_time(e1))
    step_ms = [s.elapsed_time(e) for s, e in evs]
    total_pix = cx.allsum(out_pix) if shard != "weak" else cx.world * out_pix
    res = {"ms_per_step": total_ms / steps, "value": total_pix * steps / (total_ms / 1e3) / 1e6, "unit": "Mpix/s",
           "jobs_this_rank": len(mine), "gpu_launches": int(launches), "kernel_launches_per_step": batch.launches_per_run, "steps": steps}
    achieved = algo_bytes / (float(np.mean(step_ms)) / 1e3) / 1e9
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(name)
        if tj:
            traffic = tj["traffic_bytes_per_job"] * len(mine)
    except Exception:
        traffic = None
    res["roofline"] = {"bound": "hbm", "achieved": achieved, "peak": cx.peak, "unit": "GB/s", "frac": achieved / cx.peak, "traffic": traffic,
                       "frac_of_nominal_8000": achieved / 8000.0,      # SURVEY §8d asks for both denominators
                       "peak_source": cx.peak_src, "algorithmic_bytes_per_step": int(algo_bytes), "kernel_launches_per_step": batch.launches_per_run,
                       "ms_per_launch_group": float(np.mean(step_ms)), "ms_min": float(np.min(step_ms)), "rank": cx.rank}
    if dump:
        def frame(i, rows):
            j, si, k = slots[i]
            p = plans[si]
            t = dsts[si][k, :, :p.out_w * p.out_c]
            if rows is not None:
                t = t[torch.as_tensor(rows, device=dev)]
            return j, t.reshape(-1, p.out_w, p.out_c).cpu().numpy()

        def job_shape(i):
            p = plans[slots[i][1]]
            return p.out_h, p.out_w, p.out_c
        res["_dump"] = [frame(i, rows) for i, rows in dump_sample(len(slots), job_shape)]
    batch.close()
    del srcs, dsts
    torch.cuda.empty_cache()

    # ---------------- end to end: host (pinned) buffers through the C ABI ---------------------------------
    # up to 32 distinct pinned sources per shape, cycled; every request still copies its own crop window H2D and its
    # result D2H inside the timed region. cfg5 runs a 4096-job sample of the farm (every 16th job).
    if e2e_steps > 0:
        sample = mine if len(mine) <= 4096 else mine[::max(1, len(mine) // 4096)][:4096]
        pools, outs = {}, {}
        h_plans, h_srcs, h_dsts = [], [], []
        h2d = d2h = 0
        cnt = {}
        for j in sample:
            si = order[j]
            (h, w, c), _, _ = wl["jobs"][si]
            p = plans[si]
            if si not in pools:
                n_pool = 32 if not wl.get("interleave") else 1
                pools[si] = [torch.randint(0, 256, (h, w, c), dtype=torch.uint8).pin_memory() for _ in range(n_pool)]
                outs[si] = [torch.empty((p.out_h, p.out_w, p.out_c), dtype=torch.uint8).pin_memory() for _ in range(n_pool)]
            k = cnt.get(si, 0); cnt[si] = k + 1
            h_plans.append(p); h_srcs.append(pools[si][k % len(pools[si])].numpy()); h_dsts.append(outs[si][k % len(outs[si])].numpy())
            x, y, ww, hh = p.window
            h2d += ww * hh * c; d2h += p.out_w * p.out_h * p.out_c
        hj = api.HostJobs(h_plans, h_srcs, h_dsts)
        e2e_pix = sum(p.out_w * p.out_h for p in h_plans)
        hj.run(L, n_streams=4)                                         # warm-up: allocates the lanes
        l0 = L.launch_count()
        times = []
        for _ in range(e2e_steps):
            cx.barrier()
            t0 = time.perf_counter()
            hj.run(L, n_streams=4)
            torch.cuda.synchronize()
            times.append(cx.allmax(time.perf_counter() - t0))
        e2e_launches = (L.launch_count() - l0) // max(1, e2e_steps)
        tot_pix = cx.allsum(e2e_pix) if shard != "weak" else cx.world * e2e_pix
        med = statistics.median(times)
        res["e2e"] = {"value": tot_pix / med / 1e6, "unit": "Mpix/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                      "jobs_per_step": len(h_plans), "steps": e2e_steps, "best": tot_pix / min(times) / 1e6, "worst": tot_pix / max(times) / 1e6,
                      "kernel_launches_per_step": int(e2e_launches), "h2d_gbs_this_rank": h2d / med / 1e9}
        # the same call with PAGEABLE frames (what cvDecodeImage / cvCreateImage hand RunJob): every window passes through the
        # lanes' pinned staging on the host cores first, every result back out of it. A 64-job sample.
        if name != "cfg5":
            m = min(64, len(h_plans))
            pg_src, pg_dst = {}, {}
            ps, pd = [], []
            for k in range(m):
                a, b = h_srcs[k], h_dsts[k]
                if id(a) not in pg_src and len(pg_src) < 16: pg_src[id(a)] = np.array(a, copy=True)
                if id(b) not in pg_dst and len(pg_dst) < 16: pg_dst[id(b)] = np.empty_like(b)
                ps.append(pg_src.get(id(a), next(iter(pg_src.values())) if pg_src else a))
                pd.append(pg_dst.get(id(b), next(iter(pg_dst.values())) if pg_dst else b))
            pj = api.HostJobs(h_plans[:m], ps, pd)
            pj.run(L, n_streams=4)
            pt = []
            for _ in range(max(3, e2e_steps // 2)):
                cx.barrier()
                t0 = time.perf_counter(); pj.run(L, n_streams=4); pt.append(cx.allmax(time.perf_counter() - t0))
            ppix = cx.world * sum(p.out_w * p.out_h for p in h_plans[:m])
            res["e2e"]["pageable_frames"] = {"value": ppix / statistics.median(pt) / 1e6, "unit": "Mpix/s", "jobs_per_step": m,
                                             "what": "same call, pageable numpy frames in and out (staged through pinned memory by the library's copy workers)"}
            del pj, ps, pd, pg_src, pg_dst
        res["_host"] = (h_plans, h_srcs, h_dsts, pools, outs)           # kept for the latency / farm legs of the caller
    res["_plans"] = plans
    res["_wl"] = wl
    return res


def request_latency(cx: Ctx, name: str):
    """One request at a time, host frame in, host frame out (pageable numpy buffers, like a decoded IplImage):
    warm plan through imp_gpu_run_host; the full operator sequence of RunJob (imp_Crop .. imp_FlushAll) repeated (plan
    cache hit) and with the plan cache emptied before each request (cold: validation, lowering, blob upload, tensor map)."""
    api, L = cx.api, cx.L
    wl = workload(name, 1)
    (h, w, c), rq, _ = wl["jobs"][0]
    cfg = api.Config(**dict(wl["cfg"], max_w=0, max_h=0))
    rng = np.random.default_rng(99)
    frames = [rng.integers(0, 256, (h, w, c), dtype=np.uint8) for _ in range(4)]
    plan = L.plan(w, h, c, cfg, **rq)
    out = np.empty((plan.out_h, plan.out_w, plan.out_c), np.uint8)
    def timed(fn, n, skip=3):
        ts = []
        for k in range(n):
            t0 = time.perf_counter(); fn(k); ts.append((time.perf_counter() - t0) * 1e3)
        ts = sorted(ts[skip:])
        return {"p50": ts[len(ts) // 2], "min": ts[0], "max": ts[-1], "n": len(ts)}
    warm = timed(lambda k: plan.run_host(frames[k % 4], out), 40, 8)
    torch = cx.torch
    pin = [torch.from_numpy(f).pin_memory() for f in frames]
    pout = torch.empty((plan.out_h, plan.out_w, plan.out_c), dtype=torch.uint8).pin_memory()
    warm_pinned = timed(lambda k: plan.run_host(pin[k % 4].numpy(), pout.numpy()), 40, 8)
    ops = api.OpsLayer(L)
    kw = dict(crop=rq.get("crop"), resize=rq.get("resize"), filters=rq.get("filters", []), simple=bool(rq.get("simple")))
    def seq(k, rq_kw):
        code, o = ops.request([frames[k % 4]], cfg, **rq_kw)
        assert code == 0
    repeat = timed(lambda k: seq(k, kw), 30, 6)
    # cold: the SAME request with the plan cache emptied before every request (outside the timed region), so each one pays
    # validation, lowering, table upload and tensor-map encode again — like for like against the repeated request
    plan.close()
    ts = []
    for k in range(12):
        L.plan_cache_clear()
        t0 = time.perf_counter(); seq(k, kw); ts.append((time.perf_counter() - t0) * 1e3)
    ts = sorted(ts[2:])
    cold_t = {"p50": ts[len(ts) // 2], "min": ts[0], "max": ts[-1], "n": len(ts)}
    return {"what": "pageable host frame in, host frame out, one request at a time (ms)",
            "run_host_warm_plan": warm, "run_host_warm_plan_pinned_frames": warm_pinned, "ops_sequence_repeat": repeat, "ops_sequence_cold_plan": cold_t,
            "cold_over_repeat": cold_t["p50"] / repeat["p50"]}


def gif_album_e2e(cx: Ctx, name: str, plans, wl, steps: int):
    """cfg3 / cfg3nn as the GIF request they describe: the frames enter as PAGES (8-bit palette indices, 1 byte per pixel over
    PCIe instead of a decoded canvas's 4), are expanded into BGRA canvases on the device (LoadGIF's loop, advancedio.c:195-248)
    and feed the frame loop there — imp_gpu_gif_album_run_host, pageable pages in, pinned results out, all inside the timed
    region. Same plan, same output pixels as the e2e leg over decoded canvases (which is D2H-bound for a 2x enlargement, so
    that leg's number is this one's ceiling); `thumbnails` is the H2D-bound counterpart: the same album shrunk 4x per axis,
    through pages and through pinned decoded canvases."""
    api, L, torch = cx.api, cx.L, cx.torch
    (h, w, c), _, n = wl["jobs"][0]
    rng = np.random.default_rng(77 + cx.rank)
    pages = [dict(indices=rng.integers(0, 256, (h, w), dtype=np.uint8), left=0, top=0, dispose=1, key=int(rng.integers(0, 256)),
                  palette=rng.integers(0, 256, (256, 4), dtype=np.uint8)) for _ in range(n)]

    def timed(fn):
        fn()
        l0 = L.launch_count()
        ts = []
        for _ in range(steps):
            cx.barrier()
            t0 = time.perf_counter(); fn(); ts.append(cx.allmax(time.perf_counter() - t0))
        return statistics.median(ts), min(ts), int((L.launch_count() - l0) // max(1, steps))

    def pages_job(plan):
        outs = [torch.empty((plan.out_h, plan.out_w, plan.out_c), dtype=torch.uint8).pin_memory() for _ in range(min(n, 32))]
        return api.GifAlbumJob(L, pages, w, h, True, plan, [outs[k % len(outs)].numpy() for k in range(n)]), outs

    job, keep = pages_job(plans[0])
    med, best, launches = timed(lambda: job.run(L))
    tot = cx.world * job.out_pixels
    res = {"value": tot / med / 1e6, "unit": "Mpix/s", "h2d_bytes_per_step": job.h2d_bytes, "d2h_bytes_per_step": job.d2h_bytes,
           "jobs_per_step": n, "steps": steps, "best": tot / best / 1e6, "kernel_launches_per_step": launches,
           "what": "the same request entering as GIF pages (palette indices) instead of decoded BGRA canvases: expanded on the device"}
    # H2D-bound counterpart: thumbnails of the same album
    small = L.plan(w, h, 4, api.Config(), resize=f"{w // 4},{h // 4}", simple=(name == "cfg3nn"))
    tjob, keep2 = pages_job(small)
    tmed, _, _ = timed(lambda: tjob.run(L))
    canv = [torch.from_numpy(cv).pin_memory() for cv in L.gif_expand(pages[:32], w, h, True)]
    couts = [torch.empty((small.out_h, small.out_w, small.out_c), dtype=torch.uint8).pin_memory() for _ in range(32)]
    hj = api.HostJobs([small] * n, [canv[k % len(canv)].numpy() for k in range(n)], [couts[k % 32].numpy() for k in range(n)])
    cmed, _, _ = timed(lambda: hj.run(L, n_streams=4))
    tpix = cx.world * tjob.out_pixels
    res["thumbnails"] = {"request": f"resize={w // 4},{h // 4}", "pages": {"value": tpix / tmed / 1e6, "unit": "Mpix/s", "ms": tmed * 1e3, "h2d_bytes_per_step": tjob.h2d_bytes},
                         "decoded_pinned_canvases": {"value": tpix / cmed / 1e6, "unit": "Mpix/s", "ms": cmed * 1e3, "h2d_bytes_per_step": n * w * h * 4}}
    small.close()
    return res


def h2d_ceiling(cx: Ctx):
    """Bare pinned cudaMemcpyAsync H2D, all ranks at once: what the box gives the e2e legs to work with."""
    torch = cx.torch
    n = 32 << 20
    hs = [torch.empty(n, dtype=torch.uint8).pin_memory() for _ in range(8)]
    ds = [torch.empty(n, dtype=torch.uint8, device=cx.dev) for _ in range(8)]
    st = [torch.cuda.Stream(device=cx.dev) for _ in range(4)]
    def run(streams, reps=48):
        cx.barrier()
        t0 = time.perf_counter()
        for r in range(reps):
            with torch.cuda.stream(streams[r % len(streams)]):
                ds[r % 8].copy_(hs[r % 8], non_blocking=True)
        torch.cuda.synchronize()
        dt = cx.allmax(time.perf_counter() - t0)
        return n * reps / dt / 1e9
    run(st[:1], 8)
    one = run(st[:1]); four = run(st)
    # both directions at once (what a same-size request — cfg4, or cfg3's 4x larger results — loads the link with)
    back = [torch.empty(n, dtype=torch.uint8).pin_memory() for _ in range(4)]
    def duplex(reps=32):
        cx.barrier()
        t0 = time.perf_counter()
        for r in range(reps):
            with torch.cuda.stream(st[0]):
                ds[r % 4].copy_(hs[r % 4], non_blocking=True)
            with torch.cuda.stream(st[1]):
                back[r % 4].copy_(ds[4 + r % 4], non_blocking=True)
        torch.cuda.synchronize()
        dt = cx.allmax(time.perf_counter() - t0)
        return n * reps / dt / 1e9
    duplex(4)
    both = duplex()
    return {"what": "32 MB pinned -> device copies (8 buffers cycled), all ranks concurrently, GB/s per rank: the box's ceiling for the e2e legs",
            "one_stream": one, "four_streams": four, "aggregate_gbs": max(one, four) * cx.world,
            "duplex_each_direction": both, "duplex_what": "H2D and D2H of 32 MB buffers issued together on two streams: GB/s sustained in EACH direction"}


def strip_private(d):
    return {k: v for k, v in d.items() if not k.startswith("_")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2")
    ap.add_argument("--scale", type=int, default=1, help="divide the job count (debug only; 1 = the named workload)")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--extras", default="all", help="all | none | comma list of cfg1,cfg3,cfg3nn,cfg4,cfg5 (other BASELINE configs measured in the same run)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write a fixed sample of the frames the headline's last "
                    "step produced as DIR/<config>_job<index>.npy (float32 HxWxC; a seeded sample of the rows of a frame too large on its "
                    "own, the rows bench.dump_sample picks, in order; under 64 MB in all; rank 0), to compare two builds")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed; it does not apply to --impl reference")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    wl = workload(a.config, a.scale)
    extras = [] if a.extras == "none" else (EXTRA_ORDER if a.extras == "all" else [e for e in a.extras.split(",") if e])
    extras = [e for e in extras if e != a.config]
    cores = os.cpu_count() or 1

    # ---------------- reference arm: the CPU path, rank 0 only ------------------------------------------
    if a.impl == "reference":
        if rank != 0:
            return
        per_worker = max(1, CPU_PER_WORKER.get(a.config, 8) // 2)
        for _ in range(a.warmup):
            cpu_run(a.config, a.scale, 1, cores)
        vals, kind = [], "port"
        t_total = 0.0
        for _ in range(a.steps):
            v, kind, wall = cpu_run(a.config, a.scale, per_worker, cores)
            vals.append(v); t_total += wall
        v = float(np.mean(vals))
        sample = f"{per_worker} request(s) per worker x {cores} single-threaded worker processes per step, same request as '{a.config}'"
        print(json.dumps({"metric": METRIC, "value": v, "unit": "Mpix/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
                          "ms_per_step": 1e3 * t_total / max(1, a.steps), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": "u8 pixels, f32/i32 arithmetic", "data": "synthetic", "impl": "reference", "config": config_dict(a.config, wl),
                          "cpu_baseline": {"value": v, "unit": "Mpix/s", "cores": cores, "kind": kind, "sample": sample},
                          "e2e": {"value": v, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))
        return

    # ---------------- our arm -----------------------------------------------------------------------------
    cx = Ctx(a)
    stop, samples = threading.Event(), []
    th = threading.Thread(target=sample_clocks, args=(stop, samples), daemon=True)
    th.start()
    head = measure(cx, a.config, a.steps, a.warmup, a.e2e_steps, shard="weak", dump=bool(a.dump_outputs))
    stop.set(); th.join(timeout=2)            # clocks were sampled across the device-timed and the end-to-end regions of the headline
    if a.dump_outputs and rank == 0:
        write_dump(a.dump_outputs, a.config, head.pop("_dump"))
    ceiling = h2d_ceiling(cx)
    lat = {}
    if rank == 0:
        for nm in ([a.config] + (["cfg1"] if a.config != "cfg1" else [])):
            try:
                lat[nm] = request_latency(cx, nm)
            except Exception as ex:
                lat[nm] = {"failed": repr(ex)}
    cx.barrier()

    extra_out = {}
    for nm in extras:
        if world > 1 and nm != "cfg5":
            continue                           # N > 1: the headline (weak) and cfg5 (strong); the rest is measured at N = 1
        if nm == "cfg5" and world > 1:
            r = measure(cx, nm, max(3, a.steps // 4), a.warmup, max(3, a.e2e_steps // 3), shard="mod")
            r2 = measure(cx, nm, max(3, a.steps // 4), a.warmup, 0, shard="lpt")
            e = strip_private(r)
            e["scaling"] = "strong: the same 65,536 jobs at every N, job i on GPU i mod N (no collective on the data path)"
            e["size_aware"] = {"ms_per_step": r2["ms_per_step"], "value": r2["value"], "what": "largest-first by algorithmic bytes instead of i mod N"}
            # the library's own multi-GPU entry point, driven from ONE process: rank 0 shards a 4096-job sample of the farm
            # over all N GPUs (one host thread + 4 streams per GPU) while the other ranks wait at the barrier
            cx.cpu_barrier()
            if rank == 0:
                h_plans, h_srcs, h_dsts, pools, outs = r["_host"]
                hj = cx.api.HostJobs(h_plans, h_srcs, h_dsts)
                pix = sum(p.out_w * p.out_h for p in h_plans)
                farm = {}
                for pol, pname in ((cx.api.FARM_ROUND_ROBIN, "round_robin"), (cx.api.FARM_SIZE_AWARE, "size_aware")):
                    hj.run(cx.L, n_streams=4, n_gpus=world, policy=pol)
                    ts = []
                    for _ in range(3):
                        t0 = time.perf_counter(); hj.run(cx.L, n_streams=4, n_gpus=world, policy=pol); ts.append(time.perf_counter() - t0)
                    farm[pname] = {"value": pix / statistics.median(ts) / 1e6, "unit": "Mpix/s", "jobs": len(h_plans), "n_gpus": world}
                hj.run(cx.L, n_streams=4)
                t0 = time.perf_counter(); hj.run(cx.L, n_streams=4); t1 = time.perf_counter() - t0
                farm["one_gpu_same_jobs"] = {"value": pix / t1 / 1e6, "unit": "Mpix/s"}
                farm["what"] = "imp_gpu_farm_run_host_policy from rank 0 alone over all GPUs of the box, host frames, wall clock"
                cx.L.set_device(cx.local)
                e["farm_api"] = farm
            cx.cpu_barrier()
            extra_out[nm] = e
            continue
        # sub-millisecond steps: four times the steps, so that one host-side scheduling blip between two launches (seen once: a
        # 20-step cfg3 region of 10.5 ms measured 12.4) does not move the mean; cfg5's 70 ms steps need fewer
        st = a.steps * 4 if nm != "cfg5" else max(3, a.steps // 4)
        r = measure(cx, nm, st, a.warmup, max(3, a.e2e_steps // 2), shard="weak", seed_off=17)
        e = strip_private(r)
        e["config"] = config_dict(nm, r["_wl"])
        if nm in ("cfg3", "cfg3nn") and a.e2e_steps > 0:
            e["e2e_gif_pages"] = gif_album_e2e(cx, nm, r["_plans"], r["_wl"], max(3, a.e2e_steps // 2))
        if world == 1 and not a.no_cpu:
            e["cpu_baseline"] = cpu_baseline(nm, a.scale, cores)
        extra_out[nm] = e
        del r

    if rank != 0:
        if cx.dist is not None:
            cx.cpu_barrier()                   # rank 0 times the CPU reference on the host cores meanwhile: wait on the CPU, not on the GPU
            cx.dist.barrier(); cx.dist.destroy_process_group()
        return
    line = {
        "metric": METRIC, "value": head["value"], "unit": "Mpix/s", "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
        "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8 pixels, f32/i32 arithmetic", "data": "synthetic",
        "config": config_dict(a.config, wl),                  # the very dict the reference arm prints
        "workload_detail": {"jobs_per_gpu": head["jobs_this_rank"],
                            "e2e_inputs": "32 distinct pinned host frames per shape, cycled; each request copies its crop window H2D and its result D2H",
                            "rank_cpu_binding": "NVML cpu affinity of the rank's GPU" if cx.numa_bound else "none"},
        "e2e": head.get("e2e"),
        "gpu_launches": head["gpu_launches"],
        "roofline": head["roofline"],
        "clocks": clocks_summary(samples),
        "h2d_ceiling": ceiling,
        "request_latency_ms": lat,
        "plan_cache": cx.L.plan_cache_stats(),
        "extra_configs": extra_out,
    }
    if not a.no_cpu:
        line["cpu_baseline"] = cpu_baseline(a.config, a.scale, cores)      # at every N: the same run, the same box (north_star)
    if cx.dist is not None:
        cx.cpu_barrier()
    print(json.dumps(line))
    if cx.dist is not None:
        cx.dist.barrier(); cx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
