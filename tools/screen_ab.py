"""A/B timing of the two mma.sync screening shapes in one GPU session: one warp per item (NB_SCREEN_MMA=3) against one CTA of four warps per
item (NB_SCREEN_MMA=2).  Everything goes to the directory OUT:

  card.txt          name, power limit and max SM clock of the card
  bench.jsonl       bench.py --no-cpu --no-sides lines, the two shapes alternated, REPS runs each per workload
  profile.jsonl     per-launch time of the screen kernel (torch.profiler, a run of its own per shape): C4, full batch
  outputs_equal.txt bench.py --dump-outputs of both shapes compared with np.array_equal (S, U, D, min_distance)

    python tools/screen_ab.py --out DIR [--reps 3] [--steps 20] [--warmup 5] [--workloads C4,C3,C5] [--skip bench,profile,outputs]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = (("cta", "2"), ("warp", "3"))  # NB_SCREEN_MMA values: each shape forced


def _env(v):
    return dict(os.environ, NB_SCREEN_MMA=v)


def bench(out, workloads, reps, steps, warmup):
    with open(os.path.join(out, "bench.jsonl"), "w") as f:
        for wl in workloads:
            for rep in range(reps):
                for name, v in SHAPES:
                    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", wl, "--no-cpu", "--no-sides", "--steps", str(steps),
                                        "--warmup", str(warmup)], env=_env(v), capture_output=True, text=True, cwd=ROOT)
                    try:
                        d = json.loads(r.stdout.strip().splitlines()[-1])
                        rec = dict(workload=wl, shape=name, rep=rep, ms_per_step=d["ms_per_step"], dune_kernel_ms=d.get("roofline", {}).get("kernel_ms"))
                    except Exception:
                        rec = dict(workload=wl, shape=name, rep=rep, error=(r.stderr or r.stdout)[-400:])
                    print(json.dumps(rec), flush=True)
                    f.write(json.dumps(rec) + "\n")


PROFILE = r"""
import json, os, sys
sys.path.insert(0, os.path.join(sys.argv[1], "tests")); sys.path.insert(0, sys.argv[1])
import torch
from torch.profiler import profile, ProfilerActivity
from gpu_helpers import make_pan, to_cuda
from helpers import CONFIGS, make_inputs
cfg = CONFIGS["C4"]
inp = to_cuda(make_inputs(cfg, B=cfg.B))
pan = make_pan(cfg, max_envs=cfg.B, overlap=2)
with torch.no_grad():
    for _ in range(3):
        pan(inp["nom_s"], inp["nom_u"], inp["ref_s"], inp["ref_us"], inp["points"], inp["velocities"])
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            pan(inp["nom_s"], inp["nom_u"], inp["ref_s"], inp["ref_us"], inp["points"], inp["velocities"])
        torch.cuda.synchronize()
res = {}
for e in prof.key_averages():
    if "dune_screen" in e.key or "dune_refine" in e.key or "nrmp" in e.key.lower():
        res[e.key[:60]] = dict(count=e.count, us_per_launch=e.device_time_total / max(1, e.count), us_total_per_step=e.device_time_total / 5)
print(json.dumps(dict(shape=sys.argv[2], kernels=res)))
"""


def profile_screen(out):
    with open(os.path.join(out, "profile.jsonl"), "w") as f:
        for name, v in SHAPES:
            r = subprocess.run([sys.executable, "-c", PROFILE, ROOT, name], env=_env(v), capture_output=True, text=True, cwd=ROOT)
            line = r.stdout.strip().splitlines()[-1] if r.returncode == 0 else json.dumps(dict(shape=name, error=r.stderr[-400:]))
            print(line, flush=True)
            f.write(line + "\n")


def outputs_equal(out, workloads):
    import numpy as np

    lines = []
    for wl in workloads:
        dirs = {}
        for name, v in SHAPES:
            d = os.path.join(out, f"dump_{wl}_{name}")
            subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", wl, "--no-cpu", "--no-sides", "--steps", "2", "--warmup", "3",
                            "--dump-outputs", d], env=_env(v), capture_output=True, text=True, cwd=ROOT, check=True)
            dirs[name] = d
        for f in sorted(os.listdir(dirs["cta"])):
            a, b = np.load(os.path.join(dirs["cta"], f)), np.load(os.path.join(dirs["warp"], f))
            lines.append(f"{wl} {f}: shape {a.shape} array_equal={np.array_equal(a, b, equal_nan=True)}")
    with open(os.path.join(out, "outputs_equal.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workloads", default="C4,C3,C5")
    ap.add_argument("--out", required=True, help="output directory (created if missing)")
    ap.add_argument("--skip", default="", help="comma list of parts to leave out: bench, profile, outputs")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    skip = set(args.skip.split(","))
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True).stdout
    with open(os.path.join(args.out, "card.txt"), "w") as f:
        f.write(card)
    print(card, flush=True)
    wls = [w for w in args.workloads.split(",") if w]
    if "outputs" not in skip:
        outputs_equal(args.out, wls)
    if "bench" not in skip:
        bench(args.out, wls, args.reps, args.steps, args.warmup)
    if "profile" not in skip:
        profile_screen(args.out)


if __name__ == "__main__":
    main()
