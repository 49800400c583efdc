#!/usr/bin/env python
"""bench.py -- PAN control steps/sec on the BASELINE.json north-star workload.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload C4] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

A "step" = one batched PAN.forward (iter_num fixed at the config's K by iter_threshold = 0) over
B environments per GPU (weak scaling: every rank owns B envs of the same seeded family, env ids
offset by rank*B; at the end of each step the per-env trajectories are gathered with one NCCL
all_gather, inside the timed region).  Prints ONE JSON line (rank 0).

  value ...... env-steps/s, inputs resident in HBM, device-timed (CUDA events, max over ranks)
  e2e ........ same metric through the public API with pinned HOST tensors (H2D + D2H inside)
  roofline ... DUNE kernel (the dominant launch): algorithmic GEMM FLOPs / CUDA-event duration
  cpu_baseline the CPU oracle (port of the reference path) on the box's host cores, bounded sample

--impl reference times that CPU path alone, on all host cores (rank 0 only).

--dump-outputs DIR (C1 ... C5, --impl ours) writes what the last timed step returned -- the trajectories S, U, D and
min_distance of every environment, unpacked from ShardedPAN.step -- as float32 DIR/<name>.npy, so that two builds run with
the same arguments (hence the same seeded inputs) can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

METRIC = "PAN control steps/sec (batched envs, T x N x K)"
DUMP_LIMIT_BYTES = 64 << 20
UNIT = "env-steps/s"
F_PT = 8576  # GEMM FLOPs per point-step at E=4: 2*(2*32 + 4*32*32 + 32*4)   (SURVEY.md 8d)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        z = json.load(open(path))
        return dict(hbm_gbs=z["hbm_gbs"], tflops=z["bf16_tflops_sustained"], which="measured (MEASURED_PEAKS.json, sustained bf16)")
    return dict(hbm_gbs=6650.0, tflops=1400.0, which="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=reasons, samples=len(sm))


# --------------------------------------------------------------------------------------------
# CPU path (the oracle port of the reference: oracle/pan.py) -- cpu_baseline and --impl reference
# --------------------------------------------------------------------------------------------
def cpu_quota_cores():
    """CPU-time quota of this container in cores (cgroup v2 cpu.max / v1 cfs quota), or None when unlimited.
    The round-2 GPU box showed 128 logical CPUs in its affinity mask but handed 128 busy workers only ~16 cores of
    CPU time (wall-clock rate 95 env-steps/s, rate from the workers' own CPU time 760): the quota is what counts."""
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        return None if q == "max" else float(q) / float(p)
    except (OSError, ValueError):
        pass
    try:
        q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        p = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        return None if q <= 0 else q / p
    except (OSError, ValueError):
        return None


def host_cores() -> int:
    """Worker processes to start = cores this process can actually use: affinity mask, capped by the cgroup CPU quota."""
    try:
        n = max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        n = os.cpu_count() or 1
    q = cpu_quota_cores()
    if q is not None:
        n = max(1, min(n, int(q + 0.5)))
    return n


def _cpu_worker(args):
    """One task = a list of environments run one after the other through the CPU oracle (oracle/pan.py).
    A failing environment is counted, never fatal (round 1 lost the whole arm to one Cholesky failure)."""
    cname, env_ids, K, thr = args
    import torch

    torch.set_num_threads(1)
    from helpers import CONFIGS, make_inputs, oracle_factory

    cfg = CONFIGS[cname]
    mk = oracle_factory(cfg, K=K, iter_threshold=thr)
    out = dict(envs=0, failed=0, fallbacks=0, t_dune=0.0, t_nrmp=0.0, iters=0, wall=0.0, cpu=0.0)
    t0, c0 = time.perf_counter(), time.process_time()
    for e in env_ids:
        inp = make_inputs(cfg, B=1, env_offset=e)
        pan = mk()
        vel = None if inp["velocities"] is None else inp["velocities"][0]
        try:
            pan.forward(inp["nom_s"][0], inp["nom_u"][0], inp["ref_s"][0], inp["ref_us"][0], inp["points"][0], vel)
            out["envs"] += 1
        except Exception:  # noqa: BLE001 -- reported as a count
            out["failed"] += 1
        out["fallbacks"] += pan.fallbacks
        out["t_dune"] += pan.t_dune
        out["t_nrmp"] += pan.t_nrmp
        out["iters"] += pan.iters_run
    out["wall"], out["cpu"] = time.perf_counter() - t0, time.process_time() - c0
    return out


class CpuPool:
    """Persistent worker processes (one per usable core, one thread each); start-up and imports are paid
    once in a warm-up task so that the timed region only contains oracle work."""

    def __init__(self, cname: str, K: int, procs: int, iter_threshold: float = 0.0):
        import multiprocessing as mp

        for var in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
            os.environ[var] = "1"  # inherited by the spawned workers
        self.cname, self.K, self.procs, self.thr = cname, K, procs, iter_threshold
        self.pool = mp.get_context("spawn").Pool(procs)
        # warm-up: imports, page-in, one full-K environment per worker (first-call costs of torch / scipy)
        self.pool.map(_cpu_worker, [(cname, [10 ** 6 + i], K, iter_threshold) for i in range(procs)], chunksize=1)

    def run(self, n_envs: int, first_env: int = 0) -> dict:
        """n_envs environments spread round-robin over the workers; returns wall-clock rate and the split."""
        chunks = [list(range(first_env + i, first_env + n_envs, self.procs)) for i in range(self.procs)]
        chunks = [c for c in chunks if c]
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_worker, [(self.cname, c, self.K, self.thr) for c in chunks], chunksize=1)
        wall = time.perf_counter() - t0
        tot = {k: sum(r[k] for r in res) for k in res[0]}
        done = max(1, tot["envs"])
        return dict(rate=tot["envs"] / wall, wall=wall, envs=tot["envs"], failed=tot["failed"], fallbacks=tot["fallbacks"],
                    dune_ms_per_env=1e3 * tot["t_dune"] / done, nrmp_ms_per_env=1e3 * tot["t_nrmp"] / done, iters_per_env=tot["iters"] / done,
                    # throughput the same work would reach if every worker had a core to itself all the time: a wall-clock
                    # rate far below it means the host was shared / oversubscribed during the sample
                    rate_from_cpu_time=len(chunks) * tot["envs"] / max(tot["cpu"], 1e-9), slowest_worker_s=max(r["wall"] for r in res))

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_sample(cname: str, K: int, iter_threshold: float, rounds: int, envs_per_worker: int, first_env: int = 0):
    """`rounds` back-to-back samples of envs_per_worker x cores environments; returns (summary dict, per-round list)."""
    cores = host_cores()
    pool = CpuPool(cname, K, cores, iter_threshold)
    per_round = cores * envs_per_worker
    runs = [pool.run(per_round, first_env=first_env + i * per_round) for i in range(rounds)]
    pool.close()
    rates = [r["rate"] for r in runs]
    walls = [r["wall"] for r in runs]
    envs = sum(r["envs"] for r in runs)
    mean = lambda key: float(sum(r[key] * r["envs"] for r in runs) / max(1, envs))
    summary = dict(value=envs / sum(walls), cores=cores, rounds=rounds, envs_per_round=per_round, envs=envs,
                   failed_envs=sum(r["failed"] for r in runs), highs_fallback_solves=sum(r["fallbacks"] for r in runs),
                   rate_per_round=rates, spread=(max(rates) - min(rates)) / max(rates) if rates else None, wall_s=sum(walls),
                   dune_ms_per_env=mean("dune_ms_per_env"), nrmp_ms_per_env=mean("nrmp_ms_per_env"), pan_iterations_per_env=mean("iters_per_env"),
                   env_steps_per_s_per_core=envs / sum(walls) / cores, rate_from_cpu_time=float(np.mean([r["rate_from_cpu_time"] for r in runs])),
                   effective_cores=float(np.mean([r['rate'] / max(r['rate_from_cpu_time'], 1e-9) for r in runs])) * cores, logical_cpus=os.cpu_count(), affinity_cpus=len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else None, cgroup_quota_cores=cpu_quota_cores())
    return summary, runs


CPU_WHAT = ("oracle/pan.py: the reference's torch-CPU DUNE code restated (pinned bit-for-bit to the reference) + float64 interior point "
            "solve of the reference's program in place of cvxpylayers/ECOS (not installable here); one process per core, one thread each")


def run_reference(args):
    """--impl reference: the CPU path alone on all usable host cores.  A step = 8 environments per core (one full pass of the
    hot path, K PAN iterations, per environment); at most 4 timed steps so that the driver's --steps 20 ends within minutes."""
    from helpers import CONFIGS

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = CONFIGS[args.workload]
    steps = max(1, min(args.steps, 4))
    summ, runs = cpu_sample(args.workload, cfg.K, args.iter_threshold, steps, 8)
    ms = 1e3 * summ["wall_s"] / steps
    value = summ["value"]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=max(args.gpus, world), steps=steps, warmup=1, ms_per_step=ms, higher_is_better=True,
                scaling="weak", vs_baseline=None, dtype="f32 (MLP) / f64 (QP)", data="synthetic", impl="reference",
                config=dict(workload=f"{args.workload} {cfg.name}: T={cfg.T} N={cfg.N} K={cfg.K} M={cfg.M} dyn={cfg.dynamic}", envs_per_step=summ["envs_per_round"],
                            note="CPU arm: throughput does not depend on the GPU count; rank 0 alone runs it"),
                cpu_baseline=dict(value=value, unit=UNIT, cores=summ["cores"], kind="port",
                                  sample=f"{summ['envs_per_round']} envs/step x {steps} steps of {args.workload} (8 envs per worker process, {summ['cores']} processes, warm-up = 1 env per worker); {CPU_WHAT}",
                                  **{k: summ[k] for k in ("failed_envs", "highs_fallback_solves", "rate_per_round", "spread", "dune_ms_per_env", "nrmp_ms_per_env",
                                                           "pan_iterations_per_env", "env_steps_per_s_per_core", "rate_from_cpu_time", "logical_cpus", "affinity_cpus",
                                                           "cgroup_quota_cores", "effective_cores")}),
                e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------
class PanBench:
    """One workload on this rank's GPU: B_local environments (global batch = sum over ranks), two rotating input
    sets (distinct environments) + a 256 MiB L2 flush between timed steps.  Every step -- device-resident or from
    pinned host memory -- goes through neupan_b200.parallel.ShardedPAN (PAN.forward + the one all_gather)."""

    def __init__(self, cname, B_local, env_base, dev, world, total, args, iter_threshold=0.0, flush=None):
        import torch

        from gpu_helpers import make_pan
        from helpers import CONFIGS, make_inputs
        from neupan_b200 import _lib
        from neupan_b200.parallel import ShardedPAN

        self.torch, self.cfg, self.B, self.dev, self.world, self.total = torch, CONFIGS[cname], B_local, dev, world, total
        cfg = self.cfg
        self.n_sets = 2
        sets = []
        for s_ in range(self.n_sets):
            inp = make_inputs(cfg, B=B_local, env_offset=env_base + s_ * total)
            sets.append({k: (None if v is None else torch.from_numpy(v)) for k, v in inp.items()})
        self.dsets = [{k: (None if v is None else v.to(dev)) for k, v in s_.items()} for s_ in sets]
        self.hsets = [{k: (None if v is None else v.pin_memory()) for k, v in s_.items()} for s_ in sets]
        self.flush = flush if flush is not None else torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
        self.pan = make_pan(cfg, K=cfg.K, iter_threshold=iter_threshold, max_envs=B_local, overlap=args.overlap, dune_kernel=args.dune_kernel, nrmp_warm=args.nrmp_warm)
        self.sp = ShardedPAN(self.pan, total)
        self.lib = _lib.load()

    def step(self, i, host=False):
        d = (self.hsets if host else self.dsets)[i % self.n_sets]
        with self.torch.no_grad():  # inference (with autograd recording PAN.forward runs in differentiable mode, like cvxpylayers would)
            return self.sp.step(d["nom_s"], d["nom_u"], d["ref_s"], d["ref_us"], d["points"], d["velocities"])

    def barrier(self):
        import torch.distributed as dist

        if self.world > 1:
            dist.barrier()
        self.torch.cuda.synchronize()

    def reduce_max(self, x: float) -> float:
        import torch.distributed as dist

        t = self.torch.tensor([x], device=self.dev, dtype=self.torch.float64)
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def time_device(self, steps, warmup):
        """(ms per step: CUDA events on the launching stream, mean over steps, max over ranks; launches per step)."""
        torch = self.torch
        for i in range(warmup):
            self.flush.zero_()
            self.step(i)
        self.barrier()
        l0 = self.lib.nb_launch_count()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        self.barrier()
        for i in range(steps):
            self.flush.zero_()  # L2 flush, outside the per-step events
            ev[i][0].record()
            self.last_out = self.step(i)
            ev[i][1].record()
        self.barrier()
        launches = (self.lib.nb_launch_count() - l0) // max(1, steps)
        ms = self.reduce_max(sum(a.elapsed_time(b) for a, b in ev) / steps)
        return ms, int(launches)

    def time_e2e(self, steps):
        """Pinned host inputs -> H2D -> PAN -> all_gather -> D2H of the gathered result, wall clock around synchronised steps."""
        for i in range(2):
            self.step(i, host=True)
        self.barrier()
        t0 = time.perf_counter()
        for i in range(steps):
            self.step(i, host=True)  # ends with a stream synchronise (the result is on the host)
        ms = (time.perf_counter() - t0) * 1e3 / steps
        return self.reduce_max(ms)

    def bytes_per_step(self):
        cfg, B, T = self.cfg, self.B, self.cfg.T
        h2d = 4 * B * (2 * 3 * (T + 1) + 2 * T + T + (2 * cfg.N) * (2 if cfg.dynamic else 1))
        d2h = 4 * self.total * (3 * (T + 1) + 2 * T + T + 1)
        return h2d, d2h

    def close(self):
        self.pan.close()


def dump_outputs(dirname, packed, T):
    """S, U, D, min_distance of one step (the packed (envs, 64) result of ShardedPAN.step) as float32 .npy files; above
    DUMP_LIMIT_BYTES a fixed seeded sample of environments, whose indices go to env_index.npy."""
    from neupan_b200.parallel import unpack_results

    os.makedirs(dirname, exist_ok=True)
    packed = packed.float().cpu()
    n = packed.shape[0]
    keep = DUMP_LIMIT_BYTES // (4 * packed.shape[1] + 8)
    if n > keep:
        idx = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        packed = packed[idx]
        np.save(os.path.join(dirname, "env_index.npy"), idx.astype(np.float64))
    for name, a in zip(("S", "U", "D", "min_distance"), unpack_results(packed, T)):
        np.save(os.path.join(dirname, f"{name}.npy"), np.ascontiguousarray(a.numpy(), np.float32))


def run_ours(args):
    import torch
    import torch.distributed as dist

    from helpers import CONFIGS
    from neupan_b200 import _lib
    from neupan_b200.parallel import shard_range

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg = CONFIGS[args.workload]
    B = args.envs or cfg.B
    T, N, K = cfg.T, cfg.N, cfg.K
    per_env = 3 * (T + 1) + 2 * T + T + 1
    lib = _lib.load()

    # ---- headline: weak scaling, B environments per GPU, K iterations forced (iter_threshold = 0) ----------------
    hb = PanBench(args.workload, B, rank * B, dev, world, world * B, args, iter_threshold=args.iter_threshold)
    sampler = ClockSampler(local)
    for i in range(2):
        hb.step(i)
    hb.barrier()
    if rank == 0:
        sampler.start()
    ms, launches = hb.time_device(args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    status_bad = int((hb.pan.status != 0).sum().item())
    iters_mean = float(hb.pan.iterations.float().mean().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, hb.last_out, T)
    e2e_ms = hb.time_e2e(args.steps)
    h2d, d2h = hb.bytes_per_step()
    pan, flush, dsets = hb.pan, hb.flush, hb.dsets

    # ---- roofline of the dominant kernel (DUNE), CUDA events around back-to-back launches ----------
    roof = None
    if rank == 0:
        import ctypes as C

        d = dsets[0]
        p = lambda x: None if x is None else C.c_void_p(x.data_ptr())
        md = torch.empty(B, device=dev)
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        reps = 5
        for _ in range(2):
            _lib.check(lib.nb_dune_forward(pan._handle, B, N, p(d["nom_s"]), p(d["points"]), p(d["velocities"]), None, p(md), st))
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tot = 0.0
        for r in range(reps):
            flush.zero_()
            a.record()
            _lib.check(lib.nb_dune_forward(pan._handle, B, N, p(d["nom_s"]), p(d["points"]), p(d["velocities"]), None, p(md), st))
            b.record()
            torch.cuda.synchronize()
            tot += a.elapsed_time(b)
        dune_ms = tot / reps
        flops = float(F_PT) * B * (T + 1) * N
        pk = peaks()
        ach = flops / (dune_ms * 1e-3) / 1e12
        alg_bytes = 4.0 * B * ((2 * N) * (2 if cfg.dynamic else 1) + 3 * (T + 1)) + 4.0 * B * (T + 1) * cfg.M * 9
        # executed tensor work (3 passes of the fp16 hi/lo split): per 128-point tile 4 layers x 6 UMMA (128x32x16) + head 6 UMMA (128x16x16)
        if args.dune_kernel == 4:
            tiles = B * (T + 1) * ((N + 127) // 128)
            exec_flops = tiles * 5 * 3 * 2.0 * 128 * 32 * 16  # screening pass: bias product + one fp16 pass (2 UMMA 128x32x16) per layer; + ~7 % for the refined candidates
            kname = ("dune_screen_mma_kernel + dune_refine_kernel + dune_tcp_kernel (single-pass fp16 interval screening of all points on mma.sync m16n8k16 with "
                     "the activations in registers; tcgen05.mma kind::f16 fp16 hi/lo 3-pass exact network for the <= 32 candidates per item and the full kernel "
                     "for the items the screen cannot narrow down; bit-identical selection to the full kernel; SASS HMMA.16816 / MUFU.TANH, UTCHMMA / LDTM / STTM)")
        elif args.dune_kernel == 3:
            tiles = B * (T + 1) * ((N + 127) // 128)
            exec_flops = tiles * 5 * 7 * 2.0 * 128 * 32 * 16
            kname = "dune_tc8_kernel (tcgen05.mma kind::f16, A from TMEM, fp16 hi/lo split, 3 passes + bias product; two threads per point = 8 warps per 128-point tile, two tiles in flight per CTA; SASS UTCHMMA / LDTM / STTM)"
        elif args.dune_kernel == 2:
            tiles = B * (T + 1) * ((N + 127) // 128)
            exec_flops = tiles * 5 * 7 * 2.0 * 128 * 32 * 16  # 5 dense layers x (bias product + 6 UMMA 128x32x16)
            kname = "dune_tcp_kernel (tcgen05.mma kind::f16, A from TMEM, fp16 hi/lo split, 3 passes + bias product; two tiles in flight per CTA; FFMA2/FHFMA epilogues; SASS UTCHMMA / LDTM / STTM)"
        else:
            tiles = B * (T + 1) * ((N + 31) // 32 * 2 + 1)
            exec_flops = tiles * (4 * 24 + 6) * 2.0 * 16 * 8 * 16
            kname = "dune_mma_kernel (mma.sync m16n8k16 f16, hi/lo split, 3 passes; SASS HMMA.16816.F32)" if args.dune_kernel == 1 else "dune_kernel (all-FP32 FFMA reference variant)"
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "dune_traffic.json")
        if os.path.exists(tpath):
            traffic = json.load(open(tpath)).get(args.workload)
        roof = dict(bound="tensor", achieved=ach, peak=pk["tflops"], unit="TFLOP/s", frac=ach / pk["tflops"], traffic=traffic,
                    kernel=kname, kernel_ms=dune_ms,
                    # a full launch (all T+1 steps) is timed; inside a control step the launches of PAN iterations k > 0 skip the step-0 items
                    share_of_step=(1.0 + max(0.0, iters_mean - 1.0) * (T / (T + 1.0) if args.dune_kernel == 4 else 1.0)) * dune_ms / ms, peak_source=pk["which"],
                    algorithmic_flops_per_launch=flops, tensor_executed_tflops=exec_flops / (dune_ms * 1e-3) / 1e12,
                    algorithmic_bytes_per_launch=alg_bytes, hbm_gbs_if_bytes_only=alg_bytes / (dune_ms * 1e-3) / 1e9, hbm_peak_gbs=pk["hbm_gbs"],
                    note="compute-bound path (SURVEY 8d): HBM < 1% utilised; the GEMMs are 32-wide slices between per-point LayerNorm/tanh, "
                         "so the kernel is bound by instruction issue / dependent-issue latency and the MUFU pipe, not by the tensor pipe -- DESIGN.md 3.1")
    hb.close()
    del hb, pan, dsets

    # ---- what BASELINE.json asks for beside the headline (VERDICT r1 item 3) --------------------------------------
    def side(cname, total, thr=0.0, steps=5, warmup=3, e2e=False):
        """ms/step and env-steps/s of `total` environments of config cname split over all ranks (strong split when world > 1)."""
        lo, hi = shard_range(total, rank, world)
        sb = PanBench(cname, hi - lo, lo, dev, world, total, args, iter_threshold=thr, flush=flush)
        m, l = sb.time_device(steps, warmup)
        out = dict(workload=f"{cname} {sb.cfg.name}", global_batch=total, envs_per_gpu=[shard_range(total, r, world)[1] - shard_range(total, r, world)[0] for r in range(world)],
                   T=sb.cfg.T, N=sb.cfg.N, K=sb.cfg.K, iter_threshold=thr, ms_per_step=m, env_steps_per_s=total / (m * 1e-3), gpu_launches=l,
                   pan_iterations_mean=sb.reduce_max(float(sb.pan.iterations.float().mean().item())),
                   envs_with_solver_status=int(sb.reduce_max(float((sb.pan.status != 0).sum().item()))))
        if e2e:
            em = sb.time_e2e(3)
            out["e2e_ms_per_step"], out["e2e_env_steps_per_s"] = em, total / (em * 1e-3)
        sb.close()
        return out

    extra = {}
    if not args.no_sides and args.workload == "C4" and not args.envs:
        if world == 1:
            extra["configs"] = {c: side(c, CONFIGS[c].B, e2e=True) for c in ("C1", "C2", "C3", "C5")}
        else:
            # BASELINE.json configs 4 and 5 as written: the GLOBAL batch split over the GPUs (strong scaling)
            extra["strong"] = {"C4": side("C4", CONFIGS["C4"].B, e2e=True), "C5": side("C5", CONFIGS["C5"].B, e2e=True)}
        # the reference's default stop criterion (pan.py:52,243): environments leave the loop once the duals settle
        extra["iter_threshold_0.1"] = side("C4", world * B, thr=0.1)

    # ---- cpu baseline (rank 0, N = 1 only), bounded sample ------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        summ, _ = cpu_sample(args.workload, K, args.iter_threshold, rounds=3, envs_per_worker=8)
        cpu = dict(value=summ["value"], unit=UNIT, cores=summ["cores"], kind="port",
                   sample=f"3 rounds x {summ['envs_per_round']} envs of {args.workload} (K={K}; 8 envs per worker process, {summ['cores']} processes, 1 thread each, "
                          f"warm-up = 1 env per worker), {summ['wall_s']:.1f} s wall; {CPU_WHAT}",
                   **{k: summ[k] for k in ("failed_envs", "highs_fallback_solves", "rate_per_round", "spread", "dune_ms_per_env", "nrmp_ms_per_env",
                                            "pan_iterations_per_env", "env_steps_per_s_per_core", "rate_from_cpu_time", "logical_cpus", "affinity_cpus", "cgroup_quota_cores",
                                            "effective_cores")})

    if rank == 0:
        value = world * B / (ms * 1e-3)
        line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup, ms_per_step=ms,
                    higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32-accurate fp16 hi/lo split on tcgen05 tensor cores (ObsPointNet) / f64 (NRMP interior point)",
                    data="synthetic",
                    config=dict(workload=f"{args.workload} {cfg.name}: B={B}/GPU T={T} N={N} K={K} M={cfg.M} dyn={cfg.dynamic}" + (f" iter_threshold={args.iter_threshold} (early stop active)" if args.iter_threshold > 0 else ""), global_batch=world * B,
                                parallelism=f"env-sharded x{world}, one all_gather of {per_env} floats/env per step (inside the timed region, device-resident and e2e)",
                                l2="2 rotating input sets + 256 MiB flush between timed steps", scene="annulus (SURVEY 8d)"),
                    e2e=dict(value=world * B / (e2e_ms * 1e-3), unit=UNIT, h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h,
                             ms_per_step=e2e_ms, api="neupan_b200.parallel.ShardedPAN.step on pinned host tensors: nb_pan_forward_h2d (upload in env chunks on a copy stream, the first DUNE pass of a chunk starts when its points have landed) -> all_gather -> D2H of the gathered trajectories"),
                    gpu_launches=int(launches), clocks=clocks, roofline=roof, cpu_baseline=cpu, envs_with_solver_status=status_bad,
                    pan_iterations_mean=iters_mean, control_steps_per_s=world / (ms * 1e-3), **extra)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# --------------------------------------------------------------------------------------------
# --workload scan: the lidar scan -> points producer (SURVEY 8f "next" row 2), measured to the same bar
def run_scan(args):
    """B scans of R beams with per-beam velocities -> points for PAN (decimated to max_points = 500, C4's N).
    metric: scans/s; roofline: HBM (a byte-moving kernel).  Algorithmic bytes per scan: 4R (ranges) + 24 (state) read,
    per output column 8 (point) + 8 (velocity) written and 8 (velocity gather) read, 4 (count) written."""
    import time

    import torch

    from neupan_b200 import _lib, scan_to_points
    from oracle import scan as oscan

    B, R, MP = args.envs or 16384, 1080, 500
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    scan = dict(angle_min=-np.pi, angle_max=np.pi, range_min=0.1, range_max=10.0)
    off, n_sets = (0.25, 0.0, 0.1), 3
    rng = np.random.default_rng(4321)
    host = [dict(ranges=torch.from_numpy(rng.uniform(0.0, 11.5, size=(B, R)).astype(np.float32)).pin_memory(),
                 velocity=torch.from_numpy(rng.uniform(-1, 1, size=(B, 2, R)).astype(np.float32)).pin_memory(),
                 states=torch.from_numpy(np.stack([rng.uniform(-5, 5, B), rng.uniform(-5, 5, B), rng.uniform(-np.pi, np.pi, B)], 1)).pin_memory())
            for _ in range(n_sets)]
    devs = [{k: v.to(dev) for k, v in h.items()} for h in host]  # 3 x 212 MB of inputs: larger than the 126 MB L2
    lib = _lib.load()

    def step(i, from_host=False):
        d = (host if from_host else devs)[i % n_sets]
        if from_host:
            d = {k: v.to(dev, non_blocking=True) for k, v in d.items()}
        pts, vel, cnt = scan_to_points(d["states"], d["ranges"], scan, off, max_points=MP, velocity=d["velocity"])
        return (pts, vel, cnt.cpu()) if from_host else (pts, vel, cnt)

    for i in range(args.warmup):
        step(i)
    torch.cuda.synchronize()
    sampler = ClockSampler(dev.index or 0)
    sampler.start()
    l0 = lib.nb_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        out = step(i)
    e1.record()
    torch.cuda.synchronize()
    launches = lib.nb_launch_count() - l0
    ms = e0.elapsed_time(e1) / args.steps
    clocks = sampler.stop()
    n_out = float(out[2].double().mean())
    # end to end: pinned host scans in, counts read back (points stay on the device for PAN)
    for i in range(2):
        step(i, True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(i, True)
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    alg = B * (4.0 * R + 24 + n_out * 24 + 4)
    pk = peaks()
    roof = dict(bound="hbm", achieved=alg / (ms * 1e-3) / 1e9, peak=pk["hbm_gbs"], unit="GB/s", frac=alg / (ms * 1e-3) / 1e9 / pk["hbm_gbs"], traffic=None,
                kernel="scan_to_points_kernel (one CTA per scan: ballot/popc ordered compaction into a shared-memory list, FP64 transform, coalesced stores)",
                kernel_ms=ms, share_of_step=1.0, peak_source=pk["which"], algorithmic_bytes_per_launch=alg,
                note="the velocity array (8R B per scan) is only gathered at the kept beams; if it had to be streamed completely the bytes would be 3x")
    line = dict(metric="lidar scans/sec -> obstacle points (batched envs)", value=B / (ms * 1e-3), unit="scans/s", n_gpus=1, steps=args.steps, warmup=args.warmup,
                ms_per_step=ms, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64 arithmetic, f32 in/out", data="synthetic",
                config=dict(workload=f"scan: B={B} scans x R={R} beams -> max_points={MP} (decimated), velocities on", global_batch=B,
                            l2=f"{n_sets} rotating input sets of {B * R * 12 / 1e6:.0f} MB each (> L2)"),
                gpu_launches=int(launches), clocks=clocks, roofline=roof,
                e2e=dict(value=B / (e2e_ms * 1e-3), unit="scans/s", h2d_bytes_per_step=int(B * (R * 12 + 24)), d2h_bytes_per_step=int(B * 4), ms_per_step=e2e_ms,
                         api="neupan_b200.scan_to_points on pinned host tensors (points stay on the device for PAN.forward)"))
    if not args.no_cpu:
        n = min(B, 4096)
        t0 = time.perf_counter()
        oscan.scan_batch(host[0]["states"].numpy()[:n], host[0]["ranges"].numpy()[:n], scan, off, max_points=MP, velocity=host[0]["velocity"].numpy()[:n])
        wall = time.perf_counter() - t0
        line["cpu_baseline"] = dict(value=n / wall, unit="scans/s", cores=1, kind="port", sample=f"{n} scans, {wall:.1f} s wall; oracle/scan.py (the reference's per-beam Python loop restated)")
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------
# --workload ipath: check_arrive + generate_nom_ref_state for B robots (SURVEY 8f "next" row 1)
def run_ipath(args):
    """metric: env path-steps/s.  Algorithmic bytes per env and step: 24 (state) + 8T (velocities) read, the path points the
    step touches (closest-point window + T reference points, 32 B each) read, 4(3(T+1)) x 2 + 4(2T) + 4T + 12 written."""
    import time

    import torch

    from neupan_b200 import InitialPathBatch, _lib
    from oracle import ipath as oip

    B, T, NPTS = args.envs or 16384, 10, 200
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    rng = np.random.default_rng(99)

    def path(b):
        pts, x, y, th = np.empty((NPTS, 4)), 0.0, 0.0, 0.3
        step, curve = 0.4 + 0.0002 * ((b % 5) - 2), 0.02 * ((b % 7) - 3)
        for i in range(NPTS):
            pts[i] = (x, y, th, 1.0 if i < 150 else -1.0)
            g = pts[i, 3]
            x += step * np.cos(th) * g; y += step * np.sin(th) * g; th += curve
        return pts

    protos = [path(b) for b in range(35)]
    paths = [protos[b % 35] for b in range(B)]
    ipb = InitialPathBatch(T, 0.1, "diff", max_envs=B, device=dev)
    ipb.set_initial_paths(paths)
    lib = _lib.load()
    n_sets = 4
    sets = []
    for s in range(n_sets):
        k = rng.integers(0, 120, B)
        st = np.stack([np.array([protos[b % 35][k[b], 0], protos[b % 35][k[b], 1], protos[b % 35][k[b], 2]]) for b in range(B)]) + rng.normal(0, 0.02, (B, 3))
        vel = rng.uniform(-1, 1, (B, 2, T)).astype(np.float32); vel[:, 0] += 3.0
        sets.append((torch.from_numpy(st).pin_memory(), torch.from_numpy(vel).pin_memory()))
    dsets = [(a.to(dev), b.to(dev)) for a, b in sets]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def step(i, host=False):
        a, b = (sets if host else dsets)[i % n_sets]
        if host:
            a, b = a.to(dev, non_blocking=True), b.to(dev, non_blocking=True)
        out = ipb.step(a, b, 4.0)
        return out[4].cpu() if host else out

    for i in range(args.warmup):
        step(i)
    torch.cuda.synchronize()
    sampler = ClockSampler(dev.index or 0)
    sampler.start()
    l0, tot = lib.nb_launch_count(), 0.0
    for i in range(args.steps):
        flush.zero_()  # the path window of an env is re-read every step: flush L2 between timed iterations
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); step(i); e1.record()
        torch.cuda.synchronize()
        tot += e0.elapsed_time(e1)
    launches = lib.nb_launch_count() - l0
    ms = tot / args.steps
    clocks = sampler.stop()
    step(0, True); torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(i, True)
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    alg = B * (24 + 8.0 * T + 32.0 * (10 + T) + 4.0 * (6 * (T + 1) + 2 * T + T) + 12)
    pk = peaks()
    roof = dict(bound="hbm", achieved=alg / (ms * 1e-3) / 1e9, peak=pk["hbm_gbs"], unit="GB/s", frac=alg / (ms * 1e-3) / 1e9 / pk["hbm_gbs"], traffic=None,
                kernel="ipath_step_kernel (one thread per environment: sequential closest-point window + T-step rollout / reference walk in FP64)",
                kernel_ms=ms, share_of_step=1.0, peak_source=pk["which"], algorithmic_bytes_per_launch=alg,
                note="latency-bound sequential per-environment logic with FP64 trigonometry; ~1 KB of traffic per environment")
    line = dict(metric="initial-path steps/sec (check_arrive + generate_nom_ref_state, batched envs)", value=B / (ms * 1e-3), unit="env-steps/s", n_gpus=1,
                steps=args.steps, warmup=args.warmup, ms_per_step=ms, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64 arithmetic, f32 out",
                data="synthetic", config=dict(workload=f"ipath: B={B} envs, T={T}, paths of {NPTS} points with a gear switch", global_batch=B, l2="L2 flushed between timed iterations"),
                gpu_launches=int(launches), clocks=clocks, roofline=roof,
                e2e=dict(value=B / (e2e_ms * 1e-3), unit="env-steps/s", h2d_bytes_per_step=int(B * (24 + 8 * T)), d2h_bytes_per_step=int(B * 4), ms_per_step=e2e_ms,
                         api="neupan_b200.InitialPathBatch.step on pinned host tensors (trajectories stay on the device for PAN.forward)"))
    if not args.no_cpu:
        n = 512
        os_ = [oip.OracleInitialPath(T, 0.1, "diff") for _ in range(n)]
        for b, o in enumerate(os_):
            o.set_initial_path([r.reshape(4, 1).copy() for r in protos[b % 35]])
        st, vel = sets[0][0].numpy(), sets[0][1].numpy().astype(np.float64)
        t0 = time.perf_counter()
        for b, o in enumerate(os_):
            if not o.check_arrive(st[b].reshape(3, 1)):
                o.generate_nom_ref_state(st[b].reshape(3, 1), vel[b], 4.0)
        wall = time.perf_counter() - t0
        line["cpu_baseline"] = dict(value=n / wall, unit="env-steps/s", cores=1, kind="port", sample=f"{n} envs, {wall:.2f} s wall; oracle/ipath.py (the reference's numpy code restated)")
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------
# --workload control: the whole control step of B robots on the device (PlannerBatch = ipath -> scan -> PAN)
def run_control(args):
    """C4's robot / adjust values and B = 4096, K = 10, T = 10; obstacles arrive as lidar scans (R = 1080 beams with per-beam
    velocities, decimated to 500 points).  value: device-timed with scans and states resident; e2e: pinned host states + scans in,
    actions out."""
    import time

    import torch

    from helpers import CONFIGS, weights_path
    from neupan_b200 import PlannerBatch, _lib

    cfg = CONFIGS["C4"]
    B, R, N = args.envs or cfg.B, 1080, cfg.N
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    rng = np.random.default_rng(2024)
    pl = PlannerBatch(B, cfg.T, cfg.dt, 4.0, robot_kwargs=cfg.robot_kwargs, adjust_kwargs=dict(cfg.adjust), device=dev,
                      pan_kwargs=dict(iter_num=cfg.K, dune_max_num=N, nrmp_max_num=cfg.M, dune_checkpoint=weights_path(cfg.model), iter_threshold=0.0, max_points=N))

    def path(j):
        pts, x, y, th = np.empty((150, 4)), 0.0, 0.0, 0.3
        for i in range(150):
            pts[i] = (x, y, th, 1.0)
            x += 0.4 * np.cos(th); y += 0.4 * np.sin(th); th += 0.004 * (j - 8)
        return pts

    protos = [path(j) for j in range(17)]
    pl.set_initial_paths([protos[b % 17] for b in range(B)])
    scan = dict(angle_min=-np.pi, angle_max=np.pi, range_min=0.1, range_max=10.0)
    n_sets, sets = 2, []
    for s in range(n_sets):
        k = rng.integers(0, 60, B)
        st = np.stack([protos[b % 17][k[b], :3] for b in range(B)]) + rng.normal(0, 0.02, (B, 3))
        sets.append(dict(states=torch.from_numpy(st).pin_memory(), ranges=torch.from_numpy(rng.uniform(2.0, 11.5, (B, R)).astype(np.float32)).pin_memory(),
                         vel=torch.from_numpy(rng.uniform(-1, 1, (B, 2, R)).astype(np.float32)).pin_memory()))
    dsets = [{k: v.to(dev) for k, v in d.items()} for d in sets]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    lib = _lib.load()

    def step(i, host=False):
        d = (sets if host else dsets)[i % n_sets]
        if host:
            d = {k: v.to(dev, non_blocking=True) for k, v in d.items()}
        action, _ = pl.forward(d["states"], d["ranges"], scan, scan_velocity=d["vel"])
        return action.cpu() if host else action

    for i in range(args.warmup):
        step(i)
    torch.cuda.synchronize()
    sampler = ClockSampler(dev.index or 0)
    sampler.start()
    l0, tot = lib.nb_launch_count(), 0.0
    for i in range(args.steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); step(i); e1.record()
        torch.cuda.synchronize()
        tot += e0.elapsed_time(e1)
    launches = (lib.nb_launch_count() - l0) // args.steps
    ms = tot / args.steps
    clocks = sampler.stop()
    step(0, True); torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(i, True)
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    print(json.dumps(dict(metric="robot control steps/sec (initial path + scan -> points + PAN, batched envs)", value=B / (ms * 1e-3), unit="env-steps/s", n_gpus=1,
                          steps=args.steps, warmup=args.warmup, ms_per_step=ms, higher_is_better=True, scaling="weak", vs_baseline=None,
                          dtype="f64 (path, scan) / fp16 hi-lo tcgen05 (ObsPointNet) / f64 (NRMP)", data="synthetic",
                          config=dict(workload=f"control: C4 robot, B={B}, T={cfg.T}, K={cfg.K}, scans of R={R} beams -> N={N} points, velocities on", global_batch=B,
                                      l2="L2 flushed between timed iterations"),
                          gpu_launches=int(launches), clocks=clocks,
                          e2e=dict(value=B / (e2e_ms * 1e-3), unit="env-steps/s", h2d_bytes_per_step=int(B * (R * 12 + 24)), d2h_bytes_per_step=int(B * 8), ms_per_step=e2e_ms,
                                   api="neupan_b200.PlannerBatch.forward on pinned host states + scans -> actions on the host"))))


# --------------------------------------------------------------------------------------------
# --workload train: DUNE training epochs (SURVEY 8f "next" row 4)
def run_train(args):
    """metric: training epochs/s of the reference's default data set (data_size 100,000 -> 80,000 training points, batch 256 = 313
    sequential Adam steps per epoch).  value: nb_dune_train_epoch (one persistent CTA, parameters in shared memory);  cpu_baseline /
    --impl reference: the same loop in eager torch on the host cores (the restatement of dune_train.py:281-362; torch picks its threads)."""
    import torch

    from helpers import CONFIGS
    from neupan_b200 import _lib
    from neupan_b200.blocks.dune_train import DUNETrain
    from neupan_b200.blocks.obs_point_net import ObsPointNet

    rb = CONFIGS["C4"].make_robot()
    G, h = np.asarray(rb.G, np.float32), np.asarray(rb.h, np.float32).reshape(-1)
    n_total, batch = 100000, 256
    torch.manual_seed(0); np.random.seed(0)
    reference = args.impl == "reference"
    tr = DUNETrain(ObsPointNet(2, G.shape[0]), G, h, "/tmp/neupan_b200_bench_train", backend="torch" if reference else "native")
    tr.optimizer.param_groups[0]["lr"] = 5e-5
    t0 = time.perf_counter()
    pts, mu, dist = tr.generate_data_set(n_total, [-25, -25, 25, 25])
    if not reference:
        torch.cuda.synchronize()
    label_s = time.perf_counter() - t0
    n = int(n_total * 0.8)
    data = (pts[:n], mu[:n], dist[:n])
    steps = max(1, min(args.steps, 2)) if reference else args.steps
    for _ in range(1 if reference else args.warmup):
        tr.train_one_epoch(data, batch, False)
    l0 = _lib.load().nb_launch_count() if not reference else 0
    t0 = time.perf_counter()
    for _ in range(steps):
        losses = tr.train_one_epoch(data, batch, False)  # synchronises (the losses come back to the host)
    wall = time.perf_counter() - t0
    ms = 1e3 * wall / steps
    line = dict(metric="DUNE training epochs/sec (80,000 points, batch 256, Adam)", value=steps / wall, unit="epochs/s", n_gpus=1, steps=steps,
                warmup=1 if reference else args.warmup, ms_per_step=ms, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
                config=dict(workload=f"train: {n} points x 313 Adam steps per epoch, E={G.shape[0]}, labels in closed form ({label_s:.3f} s for {n_total} points)"),
                loss_after=float(sum(losses)), optimizer_steps_per_s=steps * ((n + batch - 1) // batch) / wall)
    if reference:
        line.update(impl="reference", gpu_launches=0, e2e=dict(value=steps / wall, unit="epochs/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                    cpu_baseline=dict(value=steps / wall, unit="epochs/s", cores=torch.get_num_threads(), kind="port",
                                      sample=f"{steps} epoch(s); neupan_b200.blocks.dune_train backend='torch' on the CPU = the reference's loop (dune_train.py:281-362) with closed-form labels"))
    else:
        line.update(gpu_launches=int((_lib.load().nb_launch_count() - l0) // steps),
                    e2e=dict(value=steps / wall, unit="epochs/s", h2d_bytes_per_step=4 * ((n + batch - 1) // batch), d2h_bytes_per_step=32, ms_per_step=ms,
                             api="DUNETrain.train_one_epoch(backend='native'): data resident on the device, per epoch the batch rotations go in and the four loss means come out"),
                    roofline=dict(bound="latency", achieved=None, peak=None, unit=None, frac=None, traffic=None, kernel="dune_train_epoch_kernel (1 persistent CTA)",
                                  note="313 strictly sequential optimiser steps of 20 MFLOP each: neither HBM nor a math pipe is the limit; see csrc/dune_train_kernel.cuh"))
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps (>= 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C4")
    ap.add_argument("--envs", type=int, default=0, help="override B per GPU")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-sides", action="store_true", help="skip the side measurements (other BASELINE configs / strong split / iter_threshold=0.1)")
    ap.add_argument("--dune-kernel", type=int, default=4, help="NB_OPT_DUNE_KERNEL: 0 fp32 ffma, 1 mma.sync, 2 tcgen05 (every point exactly), 3 tcgen05 (two threads per point), 4 tcgen05 with screening (default)")
    ap.add_argument("--iter-threshold", type=float, default=0.0, help="PAN stop criterion (pan.py:243); 0 forces exactly K iterations (the headline), the reference default is 0.1")
    ap.add_argument("--nrmp-warm", type=int, default=0, help="NB_OPT_NRMP_WARM: 1 = NRMP solves of PAN iterations k > 0 start from iteration k-1's solution")
    ap.add_argument("--overlap", type=int, default=2, help="env sub-batches pipelined on internal streams (NB_OPT_OVERLAP)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy (PAN workloads C1 ... C5, --impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload in ("train", "control", "ipath", "scan")):
        ap.error("--dump-outputs is implemented for the PAN workloads (C1 ... C5) with --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.workload == "train":
        run_train(args)
    elif args.workload == "control" and args.impl == "ours":
        run_control(args)
    elif args.workload == "ipath" and args.impl == "ours":
        run_ipath(args)
    elif args.workload == "scan" and args.impl == "ours":
        run_scan(args)
    elif args.workload == "scan":  # CPU arm of the scan stage: the per-beam loop of the reference, restated (oracle/scan.py)
        from oracle import scan as oscan
        rng = np.random.default_rng(4321)
        n, R, MP = 64, 1080, 500
        scan = dict(angle_min=-np.pi, angle_max=np.pi, range_min=0.1, range_max=10.0)
        ranges, vel = rng.uniform(0.0, 11.5, size=(n, R)).astype(np.float32), rng.uniform(-1, 1, size=(n, 2, R)).astype(np.float32)
        states = np.stack([rng.uniform(-5, 5, n), rng.uniform(-5, 5, n), rng.uniform(-np.pi, np.pi, n)], 1)
        times = []
        for _ in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            oscan.scan_batch(states, ranges, scan, (0.25, 0.0, 0.1), max_points=MP, velocity=vel)
            times.append(time.perf_counter() - t0)
        dt = float(np.mean(times[args.warmup:]))
        v = n / dt
        print(json.dumps(dict(metric="lidar scans/sec -> obstacle points (batched envs)", value=v, unit="scans/s", n_gpus=1, steps=args.steps, warmup=args.warmup,
                              ms_per_step=dt * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64", data="synthetic", impl="reference",
                              config=dict(workload=f"scan: R={R} beams -> max_points={MP}", scans_per_step=n),
                              cpu_baseline=dict(value=v, unit="scans/s", cores=1, kind="port", sample=f"{n} scans/step; oracle/scan.py (per-beam Python loop of neupan.py:173-281)"),
                              e2e=dict(value=v, unit="scans/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))))
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
