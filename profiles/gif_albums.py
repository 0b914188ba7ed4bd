"""What running many GIF albums in one call buys over one call per album (imp_gpu_gif_albums_run_host against a loop of
imp_gpu_gif_album_run_host), on two workloads:

  thumbs  64 albums x 24 pages of 320x240 -> resize=160,120 NN (simple) + sepia (modulate=0,0,100 + colorize=704214,0.6):
          GIF-to-GIF thumbnails, the batch server's typical GIF traffic
  cfg3    8 albums x 200 pages of 480x270 -> resize=960,540,up (cubic) + modulate=0,0,100 + colorize=704214,0.6 (bench.py's cfg3)

  python profiles/gif_albums.py [--steps 10] [--warmup 2] [--out FILE]

Pages are pageable host memory (palette indices), results go to pinned buffers (cfg3 cycles 32 per album, as bench.py does:
8 x 200 distinct 2 MB results would pin 3.3 GB). Each step times one pass of each mode, the modes alternating in one
process; a figure is the median over --steps with min and max beside it, host clock around calls that end in a device
synchronise. The results of the two modes are compared on the thumbs workload first. The card's name and power limit are
read in the same run. Without a GPU the script exits non-zero.
"""
import argparse
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import ngx_http_imgproc_b200 as M               # noqa: E402
from ngx_http_imgproc_b200 import api           # noqa: E402

SEPIA = ["modulate=0,0,100", "colorize=704214,0.6"]
WORKLOADS = [("thumbs", 64, 24, 320, 240, dict(resize="160,120", simple=True, filters=SEPIA)),
             ("cfg3", 8, 200, 480, 270, dict(resize="960,540,up", filters=SEPIA))]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else "unknown"


def pages_of(rng, cw, ch, n):
    return [dict(indices=rng.integers(0, 256, (ch, cw), dtype=np.uint8), left=0, top=0, dispose=int(rng.integers(0, 4)),
                 key=int(rng.integers(-1, 256)), palette=rng.integers(0, 256, (256, 4), dtype=np.uint8)) for _ in range(n)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    L = M.library()
    if L.device_count() < 1:
        sys.exit("no GPU: nothing to measure")
    L.init(0)
    import torch
    lines = [f"card: {card()}", f"steps {a.steps} (median, min, max), warmup {a.warmup}; pageable pages in, pinned results out"]
    rng = np.random.default_rng(5)
    for name, n_albums, n_pages, cw, ch, rq in WORKLOADS:
        plan = L.plan(cw, ch, 4, api.Config(), **rq)
        per_album = n_pages if name == "thumbs" else 32
        pinned = [[torch.empty((plan.out_h, plan.out_w, plan.out_c), dtype=torch.uint8).pin_memory().numpy() for _ in range(per_album)]
                  for _ in range(n_albums)]
        albums = [(pages_of(rng, cw, ch, n_pages), cw, ch, True, plan, [pinned[i][f % per_album] for f in range(n_pages)])
                  for i in range(n_albums)]
        singles = [api.GifAlbumJob(L, *al) for al in albums]
        batched = api.GifAlbumsJob(L, albums)
        if name == "thumbs":                                      # both modes give the same bytes
            for s in singles:
                s.run(L)
            want = [[o.copy() for o in s.outs] for s in singles]
            batched.run(L)
            assert all(np.array_equal(x, y) for s, w in zip(singles, want) for x, y in zip(s.outs, w)), "modes differ"

        def one_call_per_album():
            for s in singles:
                s.run(L)

        modes = [("one call per album", one_call_per_album), ("one call for all albums", lambda: batched.run(L))]
        for _, fn in modes:
            for _ in range(a.warmup):
                fn()
        ts = {m: [] for m, _ in modes}
        launches = {}
        for _ in range(a.steps):
            for m, fn in modes:
                l0 = L.launch_count()
                t0 = time.perf_counter()
                fn()
                ts[m].append(time.perf_counter() - t0)
                launches[m] = L.launch_count() - l0
        pix = n_albums * n_pages * plan.out_w * plan.out_h
        lines.append(f"\n{name}: {n_albums} albums x {n_pages} pages of {cw}x{ch} -> {rq}  ({plan.out_w}x{plan.out_h} results)")
        med = {}
        for m, _ in modes:
            med[m] = statistics.median(ts[m])
            lines.append(f"  {m:24s} {med[m] * 1e3:9.2f} ms  (min {min(ts[m]) * 1e3:.2f}, max {max(ts[m]) * 1e3:.2f})  "
                         f"{pix / med[m] / 1e6:8.1f} Mpix/s  {launches[m]} kernel launches")
        lines.append(f"  speed-up of one call: {med[modes[0][0]] / med[modes[1][0]]:.2f}x")
        plan.close()
    text = "\n".join(lines)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
