"""Same-box A/B of the exact integer INTER_AREA taps: the default bench.py line (without the CPU baseline) over another
build of libimp_gpu.so (the parent commit's, through IMP_GPU_LIB) and over the in-tree build, alternated for --rounds
rounds, then --dump-outputs of cfg2 and cfg5 from both builds compared byte for byte. The card's name, power limit and
top SM clock are read (read-only) in the same run. Results: profiles/r05_area_exact_int.txt.

  python profiles/area_exact_ab.py --other <the parent build's libimp_gpu.so> [--rounds 3] [--json results.json]"""
import argparse
import filecmp
import json
import os
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def bench(lib, extra):
    env = dict(os.environ)
    if lib:
        env["IMP_GPU_LIB"] = lib
    r = subprocess.run([sys.executable, "bench.py", "--gpus", "1"] + extra, cwd=ROOT, env=env, capture_output=True, text=True)
    if r.returncode != 0:
        raise SystemExit(r.stdout[-2000:] + r.stderr[-3000:])
    return json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])


def line(tag, d):
    ex = " ".join(f"{k} {v['ms_per_step']:.3f}" for k, v in sorted(d.get("extra_configs", {}).items()) if isinstance(v, dict) and "ms_per_step" in v)
    e2e_s = f" | e2e Mpix/s {d['e2e']['value']:.0f}" if "e2e" in d else ""
    return f"{tag:8s} cfg2 ms {d['ms_per_step']:.4f} frac {d['roofline']['frac']:.3f} launches {d['roofline'].get('kernel_launches_per_step')} | {ex}{e2e_s}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--other", required=True, help="the build to compare against (a libimp_gpu.so of the same ABI)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--json", help="also write every bench line of every round to this file")
    a = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print("gpu:", smi, flush=True)
    builds = [("parent", os.path.abspath(a.other)), ("new", "")]
    res = {n: [] for n, _ in builds}
    for k in range(a.rounds):
        for name, lib in builds:
            d = bench(lib, ["--no-cpu"])          # the CPU baseline does not depend on the build
            res[name].append(d)
            print(f"round {k}", line(name, d), flush=True)
    for name, _ in builds:
        ms = [d["ms_per_step"] for d in res[name]]
        print(f"{name}: cfg2 ms min {min(ms):.4f} max {max(ms):.4f} mean {sum(ms) / len(ms):.4f}")
    tmp = tempfile.mkdtemp()                       # the dumps are large: compared here, not kept
    for cfg in ("cfg2", "cfg5"):
        dirs = []
        for name, lib in builds:
            d = os.path.join(tmp, f"dump_{cfg}_{name}")
            bench(lib, ["--config", cfg, "--steps", "2", "--warmup", "1", "--extras", "none", "--no-cpu", "--dump-outputs", d])
            dirs.append(d)
        cmp = filecmp.dircmp(*dirs)
        files = sorted(os.listdir(dirs[0]))
        same = not cmp.diff_files and not cmp.left_only and not cmp.right_only and all(filecmp.cmp(os.path.join(dirs[0], f), os.path.join(dirs[1], f), shallow=False) for f in files)
        print(f"dump {cfg}: {len(files)} files, identical: {same}")
    shutil.rmtree(tmp)
    if a.json:
        with open(a.json, "w") as f:
            json.dump(res, f)


if __name__ == "__main__":
    main()
