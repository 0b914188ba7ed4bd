"""What the submit forms of the GIF, format=json and format=text calls give back to a server loop.

  python profiles/submit_overlap.py [--rounds 10] [--warmup 2] [--out FILE]

One round is one tick of a batch server's loop: this round's three calls, and the preparation of the next round's inputs.
  calls        the thumbs album set of profiles/gif_albums.py (64 albums x 24 pages of 320x240 -> resize=160,120 NN + sepia),
               a brightness batch and an ASCII batch (wide ramp) of 16 cfg1-sized frames each (1920x1080x3 -> resize=640,360)
  preparation  the decoded pages and frames of the next round copied into the buffers that round reads (two buffer sets
               alternate, so the copy never touches what the device is reading)
Synchronous: imp_gpu_gif_albums_run_host, imp_gpu_batch_brightness_host and imp_gpu_batch_ascii_host one after another, then
the preparation. Submitted: the three submits back to back, the preparation, then the three waits.
Pages, frames and results are pageable host memory. The two modes alternate round by round in one process; each figure is
the median over --rounds with min and max beside it, host clock around a whole round (every round ends when its device work
has finished). The kernel launches of a round (imp_gpu_launch_count) must be the same in both modes, and both modes must
give the same bytes. The card's name and power limit are read in the same run. Without a GPU the script exits non-zero.
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

from bench import workload                      # noqa: E402  (cfg1's shape and request)
import ngx_http_imgproc_b200 as M               # noqa: E402
from ngx_http_imgproc_b200 import api           # noqa: E402

SEPIA = ["modulate=0,0,100", "colorize=704214,0.6"]
N_ALBUMS, N_PAGES, CW, CH = 64, 24, 320, 240
N_ANSWERS = 16


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else "unknown"


class Inputs:
    """One buffer set: the album set's pages, the answer batches' frames, and the argument arrays built over them once."""

    def __init__(self, L, rng, gplan, fshape):
        self.albums = [[dict(indices=np.zeros((CH, CW), np.uint8), left=0, top=0, dispose=int(rng.integers(0, 4)),
                             key=int(rng.integers(-1, 256)), palette=rng.integers(0, 256, (256, 4), dtype=np.uint8))
                        for _ in range(N_PAGES)] for _ in range(N_ALBUMS)]
        self.job = api.GifAlbumsJob(L, [(pages, CW, CH, True, gplan) for pages in self.albums])
        self.bsrc = [np.zeros(fshape, np.uint8) for _ in range(N_ANSWERS)]
        self.asrc = [np.zeros(fshape, np.uint8) for _ in range(N_ANSWERS)]

    def prepare(self, k, page_pool, frame_pool):
        """Round k's inputs: its decoded pages and frames copied into this set's buffers."""
        i = 0
        for pages in self.albums:
            for p in pages:
                np.copyto(p["indices"], page_pool[(7 * k + i) % len(page_pool)])
                i += 1
        for j, f in enumerate(self.bsrc + self.asrc):
            np.copyto(f, frame_pool[(3 * k + j) % len(frame_pool)])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    L = M.library()
    if L.device_count() < 1:
        sys.exit("no GPU: nothing to measure")
    L.init(0)
    rng = np.random.default_rng(5)
    (fshape, frq, _), = workload("cfg1")["jobs"]
    gplan = L.plan(CW, CH, 4, api.Config(), resize="160,120", simple=True, filters=SEPIA)
    fplan = L.plan(fshape[1], fshape[0], fshape[2], api.Config(), **frq)
    fplans = [fplan] * N_ANSWERS
    page_pool = [rng.integers(0, 256, (CH, CW), dtype=np.uint8) for _ in range(97)]
    frame_pool = [rng.integers(0, 256, fshape, dtype=np.uint8) for _ in range(8)]
    sets = [Inputs(L, rng, gplan, fshape) for _ in range(2)]
    sets[0].prepare(0, page_pool, frame_pool)
    tick = [0]
    prep_times = []

    def prepare_next():
        t0 = time.perf_counter()
        sets[(tick[0] + 1) % 2].prepare(tick[0] + 1, page_pool, frame_pool)
        prep_times.append(time.perf_counter() - t0)

    def synchronous():
        s = sets[tick[0] % 2]
        s.job.run(L)
        b = L.batch_brightness(fplans, s.bsrc)
        t = L.batch_ascii(fplans, s.asrc, "wide")
        prepare_next()
        return b, t

    def submitted():
        s = sets[tick[0] % 2]
        tg = s.job.submit(L)
        tb, b = L.batch_brightness_submit(fplans, s.bsrc)
        ta, texts = L.batch_ascii_submit(fplans, s.asrc, "wide")
        prepare_next()
        for t in (tg, tb, ta):
            api.HostJobs.wait(L, t)
        return b, [x.tobytes() for x in texts]

    modes = [("synchronous", synchronous), ("submitted", submitted)]
    # both modes give the same bytes on the same inputs
    outs = {}
    for m, fn in modes:
        b, t = fn()
        outs[m] = (b.tobytes(), t, [[o.copy() for o in al] for al in sets[0].job.outs])
    assert outs["synchronous"][:2] == outs["submitted"][:2], "answers differ"
    assert all(np.array_equal(x, y) for p, q in zip(outs["synchronous"][2], outs["submitted"][2]) for x, y in zip(p, q)), "albums differ"
    ts = {m: [] for m, _ in modes}
    launches = {m: set() for m, _ in modes}
    prep_times.clear()
    for r in range(a.warmup + a.rounds):
        for m, fn in modes:
            tick[0] += 1
            l0 = L.launch_count()
            t0 = time.perf_counter()
            fn()
            dt = time.perf_counter() - t0
            if r >= a.warmup:
                ts[m].append(dt)
                launches[m].add(L.launch_count() - l0)
    prep = prep_times[2 * a.warmup:]
    assert len(launches["synchronous"]) == 1 and launches["synchronous"] == launches["submitted"], launches
    med = {m: statistics.median(v) for m, v in ts.items()}
    lines = [f"card: {card()}",
             f"rounds {a.rounds} (median, min, max), warmup {a.warmup}, the modes alternating; pageable pages, frames and results",
             f"one round: {N_ALBUMS} albums x {N_PAGES} pages of {CW}x{CH} -> resize=160,120 NN + sepia; brightness and ASCII (wide) of "
             f"{N_ANSWERS} frames each, {fshape[1]}x{fshape[0]}x{fshape[2]} -> {frq}; the next round's inputs prepared on the host",
             f"  host preparation alone     {statistics.median(prep) * 1e3:9.2f} ms  (min {min(prep) * 1e3:.2f}, max {max(prep) * 1e3:.2f})"]
    for m, _ in modes:
        lines.append(f"  {m:26s} {med[m] * 1e3:9.2f} ms per round  (min {min(ts[m]) * 1e3:.2f}, max {max(ts[m]) * 1e3:.2f})  "
                     f"{next(iter(launches[m]))} kernel launches per round")
    lines.append(f"  loop time given back by the submits: {(med['synchronous'] - med['submitted']) * 1e3:.2f} ms per round")
    gplan.close()
    fplan.close()
    text = "\n".join(lines)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
