#!/usr/bin/env python
"""Benchmark: env steps/s of the batched Meta-World step (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # our arm (one rank per GPU under torchrun for N>1)
  python bench.py --impl reference --gpus N --steps K ...  # reference arm: the CPU implementation of the same
                                                            # path on the host cores (see below), rank 0 only
  python bench.py --benchmark MT10 | ML45-train | ML45-test --envs-per-gpu 8192 ...   # BASELINE configs 3 and 5
  python bench.py --gather ...                               # + optional NCCL gather of obs/reward/flags (config 4)
  python bench.py --dump-outputs DIR ...                     # + what the last timed step returned, as DIR/<name>.npy

A "step" is one VectorEnv.step over all environments of a rank (4096 by default): per env 5 physics substeps
+ 1 forward pass + obs + reward + autoreset.

STEADY STATE.  Random-action episodes get heavier as they progress (objects get knocked into contact), so a short
timed window right after `reset()` flatters the kernel.  Before anything is timed the environments are therefore
staggered uniformly over the episode phase 0..499: env e starts with `path_len = p_e`, and 500 untimed steps are run,
during which every env truncates once (after 500 - p_e steps), autoresets, and arrives p_e steps into a genuine
episode.  Any timed window, however short, then contains autoresets and the whole early/mid/late-episode contact mix.

`value` is measured with actions and state resident in HBM (CUDA events around each mw_step launch, max over ranks);
`e2e` goes through the public numpy API (`MetaWorldVecEnv.step`) with host actions in and host obs/reward/flags/info
out every step.

Reference arm: MuJoCo / gymnasium (the reference's physics + glue) are not installed in this image and cannot
be installed offline, so `oracle/` -- the float64 CPU restatement of the same path -- is what is timed, on all
host cores (one process per core, each stepping its own envs), labelled kind="port".
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "env steps/sec MT50 batched (4096 envs/GPU) at 1/2/4/8 B200 vs CPU MuJoCo"     # BASELINE.json:metric
CPU_ARM_NOTE = ("the CPU arm is NOT MuJoCo: mujoco/gymnasium are not installed and not installable here (no network); "
                "timed instead: oracle/ (float64 C + Python restatement of the same step path, pinned to the reference's Python "
                "glue by tests/test_refpin.py; its physics is unpinned against real MuJoCo)")


def benchmark_names(benchmark):
    """-> (env type names, number of one-hot ids, kind)"""
    from metaworld_b200 import benchmarks as B
    if benchmark in ("MT10", "MT25", "MT50"):
        names = getattr(B, benchmark)
        return list(names), len(names), "mt"
    if benchmark.startswith("ML"):
        name, split = benchmark.split("-")
        return list(getattr(B, name)[split]), 0, "ml"
    return [benchmark], 1, "mt"


def algorithmic_bytes(names):
    """SURVEY.md 8(d): per env step 4*(2*nq + 4*nv + 120) bytes (fp32 state, 5 substeps fused)."""
    from metaworld_b200 import modelzoo
    from metaworld_b200.tasks import TASKS
    b = []
    for n in names:
        m = modelzoo.full_model(TASKS[n].xml)
        b.append(4 * (2 * m.nq + 4 * m.nv + 120))
    return float(np.mean(b))


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons during the timed regions.  NVML (pynvml) is polled every 10 ms, so even the driver's
    20-step window (~70 ms) gets several samples; `nvidia-smi` (one process per sample, ~50 ms) is the fallback."""

    REASONS = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.stop_flag, self.active = gpu, [], False, False
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = (pynvml, pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(gpu)))
        except Exception:
            self.nvml = None

    @staticmethod
    def _physical_index(local):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[local])
            except Exception:
                pass
        return local

    def _sample_nvml(self):
        nv, h = self.nvml
        sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        try:
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        return [float(sm), float(mx)] + [bool(r & bits[k]) for k in self.REASONS]

    def _sample_smi(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        out = subprocess.run(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        r = [x.strip() for x in out.split(",")]
        return [float(r[0]), float(r[1])] + [x.lower().startswith("active") for x in r[2:6]]

    def run(self):
        while not self.stop_flag:
            if self.active:
                try:
                    self.rows.append(self._sample_nvml() if self.nvml else self._sample_smi())
                except Exception:
                    pass
            time.sleep(0.01 if self.nvml else 0.2)

    def begin(self):
        """start of a timed region (samples outside timed regions are not kept)"""
        self.active = True

    def end(self):
        self.active = False

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock samples (nvml and nvidia-smi unavailable)"], "samples": 0}
        sm = [r[0] for r in self.rows]
        mx = [r[1] for r in self.rows]
        reasons = [n for i, n in enumerate(self.REASONS) if any(r[2 + i] for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": max(mx), "reasons": reasons, "samples": len(self.rows),
                "source": "nvml" if self.nvml else "nvidia-smi"}


# ----------------------------------------------------------------------------- CPU (oracle) timing
def _cpu_worker(args):
    names, steps, seed, partial = args
    from oracle.tasks import TASKS as OT
    from metaworld_b200 import benchmarks as B
    envs = []
    for i, n in enumerate(names):
        e = OT[n]()
        t = B.make_tasks([n], False, seed=seed + i, n_goals=1)[0].unpack()
        e.set_task_vec(t["rand_vec"], partial)
        e.reset()
        envs.append(e)
    rng = np.random.default_rng(seed)
    t0 = time.perf_counter()
    n = 0
    for s in range(steps):
        for e in envs:
            if e.curr_path_length >= e.max_path_length:
                e.reset()
            e.step(rng.uniform(-1, 1, 4).astype(np.float32))
            n += 1
    dt = time.perf_counter() - t0
    flops = sum(e.data.flops for e in envs)          # oracle/mjphys.c counts the flops of its physics passes
    return n, dt, flops


def usable_cores():
    """Host threads this process may actually use: the affinity mask capped by the cgroup CPU quota (the GPU boxes
    show 128 logical cores but cpu.max = 16 CPUs)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per))))
    except Exception:
        pass
    return max(1, n)


def cpu_baseline(names, cores, steps_per_env, seed=42, partial=False):
    """Times the CPU restatement (oracle) of the same path: `cores` processes, each with its own sub-envs; the task
    types are dealt round-robin over the processes so every type of the workload is in the sample.
    -> (env steps/s, description, physics flops per env step incl. the amortised resets)"""
    import multiprocessing as mp
    per = max(1, -(-len(names) // cores))
    jobs = [([names[(c * per + k) % len(names)] for k in range(per)], steps_per_env, seed + 1000 * c, partial) for c in range(cores)]
    t0 = time.perf_counter()
    if cores == 1:
        res = [_cpu_worker(jobs[0])]
    else:
        with mp.get_context("fork").Pool(cores) as p:
            res = p.map(_cpu_worker, jobs)
    wall = time.perf_counter() - t0
    total = sum(r[0] for r in res)
    busy = max(r[1] for r in res)
    flops = sum(r[2] for r in res) / max(1, total)
    return total / busy, f"{cores} process(es) x {per} envs x {steps_per_env} random-action steps (float64 CPU restatement, wall {wall:.1f}s)", flops


def workload_string(benchmark, names, n_full, N, kind):
    sel = ("task_select=random, goals resampled on every autoreset" if kind == "mt"
           else "task_select=pseudorandom, partially observable (goal zeroed), one goal-resampling reset (sample_tasks) before the rollout")
    return (f"{benchmark}: {len(names)} task types, {N} envs/GPU (env e has type e % {len(names)}), random actions U(-1,1)^4, "
            f"500-step episodes with SAME_STEP autoreset, {sel}, "
            f"{'one-hot obs (' + str(39 + n_full) + ' columns)' if n_full else 'obs 39 columns'}; "
            "STEADY STATE: episode phase of the envs uniform over 0..499 at the start of the timed region (500 untimed pre-roll steps, see bench.py docstring)")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import mjphys
    mjphys.build()
    names, n_full, kind = benchmark_names(args.benchmark)
    cores = usable_cores()
    vals = []
    sample = ""
    t_all = time.perf_counter()
    for _ in range(args.warmup + args.steps):
        v, sample, _ = cpu_baseline(names, cores, args.ref_steps_per_env, partial=(kind == "ml"))
        vals.append(v)
        if time.perf_counter() - t_all > 150:
            break
    vals = vals[min(args.warmup, len(vals) - 1):]
    value = float(np.mean(vals))
    per_step_envs = args.envs_per_gpu * args.gpus
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "env_steps/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * per_step_envs / value, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_string(args.benchmark, names, n_full, args.envs_per_gpu, kind),
                       "tasks": names, "envs_per_gpu": args.envs_per_gpu,
                       "reference_arm": CPU_ARM_NOTE + "; each process steps its own envs through full 500-step episodes incl. resets (every episode phase is in the sample)"},
            "cpu_baseline": {"value": value, "unit": "env_steps/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "env_steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ----------------------------------------------------------------------------- GPU arm
DUMP_LIMIT_BYTES = 64 * 1024 * 1024


def dump_outputs(path, outputs):
    """Writes the tensors `env.step_torch` returned (obs, reward, terminated, truncated, info) as float32 .npy files, so
    that two builds run with the same arguments can be compared output for output.  Above DUMP_LIMIT_BYTES a fixed,
    seeded sample of env rows is written instead, and its row indices as env_index.npy."""
    host = {k: v.float().cpu().numpy() for k, v in outputs.items()}
    n = len(next(iter(host.values())))
    row_bytes = sum(a[0].nbytes for a in host.values())
    if n * row_bytes > DUMP_LIMIT_BYTES:
        k = (DUMP_LIMIT_BYTES - 4096) // (row_bytes + 8)       # room for the float64 index and the .npy headers
        rows = np.sort(np.random.default_rng(0).choice(n, k, replace=False))
        host = {k: a[rows] for k, a in host.items()}
        host["env_index"] = rows.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for k, a in host.items():
        np.save(os.path.join(path, k + ".npy"), a)


def build_env(args, rank, local):
    from metaworld_b200.vector_env import MetaWorldVecEnv
    from metaworld_b200 import benchmarks as B
    names, n_full, kind = benchmark_names(args.benchmark)
    N = args.envs_per_gpu
    # every rank owns all task types (balanced shards, no collective on the step path); goals are the benchmark's own
    # (seed), the task-selection streams differ per rank
    tasks_all = B.make_tasks(names, kind == "ml", seed=args.seed)
    tasks = [[t for t in tasks_all if t.env_name == n] for n in names]
    kw = dict(num_envs=N, seed=args.seed + 1000 * rank, max_episode_steps=500, device=local)
    if kind == "mt":
        env = MetaWorldVecEnv(names, tasks, use_one_hot=True, num_tasks=n_full, **kw)
    else:
        env = MetaWorldVecEnv(names, tasks, task_select="pseudorandom", checkpoint_env_ids=[None] * len(names), **kw)
    return env, names, n_full, kind


def stagger(env, seed):
    """Uniform episode phases: path_len p_e in 0..499, decorrelated from the task type (env e has type e % n_types)."""
    N = env.num_envs
    p = (np.arange(N) * 500 // N)[np.random.default_rng(seed).permutation(N)]
    st = env.engine.get_state()
    st["path_len"] = p.astype(np.float32)
    env.engine.set_state(st)
    env._ep_len[:] = p
    return p


def ncu_summary():
    """Numbers that cannot be measured inside a timed run come from the committed ncu capture of this round
    (profiles/rNN_k_step_ncu_summary.csv, metric,value,unit rows); the file name is reported with them."""
    try:
        import csv as _csv, glob as _glob
        path = sorted(_glob.glob(os.path.join(ROOT, "profiles", "r*_k_step_ncu_summary.csv")))[-1]
        rows = {r[0]: (float(r[1]), r[2]) for r in _csv.reader(open(path)) if len(r) == 3 and r[1].replace(".", "").replace("-", "").replace("e", "").replace("+", "").isdigit()}
        scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        d = [v * scale.get(u, 1.0) for k, (v, u) in rows.items() if k.startswith("dram__bytes_read.sum") or k.startswith("dram__bytes_write.sum")]
        out = {"source": os.path.relpath(path, ROOT), "dram_bytes_per_launch": sum(d) if d else None}
        for k in ("sm__warps_active.avg.pct_of_peak_sustained_active", "sm__throughput.avg.pct_of_peak_sustained_elapsed",
                  "smsp__thread_inst_executed_per_inst_executed.ratio", "launch__registers_per_thread", "launch__occupancy_limit_shared_mem"):
            if k in rows:
                out[k] = rows[k][0]
        return out
    except Exception:
        return {"source": None, "dram_bytes_per_launch": None}


def run_ours(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if os.environ.get("MW_BENCH_SWAP") == "1" and world == 2:       # diagnosis: rank r on device 1 - r
        local = 1 - local
    torch.cuda.set_device(local)
    if world > 1:
        if os.environ.get("MW_BENCH_PG", "nccl") == "gloo":      # diagnosis only (scripts/gpu_2gpu_diag.sh)
            dist.init_process_group("gloo")
        else:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from metaworld_b200.engine import lib

    seed_rank = int(os.environ.get("MW_BENCH_FAKE_RANK", rank))     # diagnosis: a single process with rank r's random streams
    if seed_rank != rank:
        rank_true, rank = rank, seed_rank
    env, names, n_full, kind = build_env(args, rank, local)
    N = args.envs_per_gpu
    dev = env.device
    K, W = args.steps, args.warmup
    extra = {}
    t0 = time.perf_counter()
    env.reset()
    if kind == "ml":
        # BASELINE config 5: one goal-resampling reset of every env, (a) from the snapshot cache (what the engine does in
        # steady state), (b) raw: the reference's double-pass reset (2 x 50 x 5 substeps + reset_model) for N envs on the device
        torch.cuda.synchronize(); t1 = time.perf_counter()
        env.call("sample_tasks")
        torch.cuda.synchronize(); extra["goal_resampling_reset_ms_snapshot_cache"] = 1e3 * (time.perf_counter() - t1)
        cur = env._current_tasks()
        rv = np.zeros((N, 6)); po = np.ones(N, dtype=np.uint8)
        for e, tk in enumerate(cur):
            v = tk.unpack()["rand_vec"]; rv[e, : len(v)] = v
        nsnap = lib().mw_num_snapshots(env.engine.h)
        torch.cuda.synchronize(); t1 = time.perf_counter()
        env.engine.build_snapshots([env._slot[e % env.n_types] for e in range(N)], rv, po, precise=False)
        torch.cuda.synchronize(); extra["goal_resampling_reset_ms_raw_double_pass_f32"] = 1e3 * (time.perf_counter() - t1)
        extra["goal_resampling_reset_note"] = (f"{N} envs; raw = k_snapshot on the float32 build, one warp per env, 500 mj_step each (= 100 env steps of physics); "
                                               f"snapshot cache = host task draw + k_reset copy of the cached float64-built episode start; {nsnap} cached goals")
    phases = stagger(env, args.seed + rank)
    a_pre = np.random.default_rng(args.seed + 7 + rank).uniform(-1, 1, size=(500, N, 4)).astype(np.float32)
    for i in range(500):                      # untimed pre-roll through the public numpy API (host task streams stay in sync)
        env.step(a_pre[i])
    del a_pre
    torch.cuda.synchronize()
    setup_s = time.perf_counter() - t0
    sampler = ClockSampler(local); sampler.start()
    # ---- e2e through the numpy API: pinned H2D of actions, D2H of obs/reward/flags/info inside the timed region
    Ke = min(K, args.e2e_steps)
    a_host = (np.random.default_rng(args.seed + rank).uniform(-1, 1, size=(Ke + 2, N, 4))).astype(np.float32)
    for i in range(2):
        env.step(a_host[i])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler.begin()
    t1 = time.perf_counter()
    n_final = 0
    for i in range(Ke):
        out = env.step(a_host[2 + i])
        n_final += int((out[2] | out[3]).sum())
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t1
    sampler.end()
    # ---- device-resident: actions + state in HBM, device-side task sampler, CUDA events around every step
    gen = torch.Generator(device=dev); gen.manual_seed(args.seed + rank)
    actions = torch.rand(K + W, N, 4, device=dev, generator=gen) * 2 - 1      # resident in HBM before timing
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)                    # > 126 MB L2
    noflush = os.environ.get("MW_BENCH_NOFLUSH") == "1"        # diagnosis only (how much of a sample's tail is cold-L2 latency); the line says so
    gather = None
    if args.gather and world > 1:
        side = torch.cuda.Stream(device=dev)
        g_obs = torch.empty(world * N, env.obs_dim, device=dev); g_small = torch.empty(world * N, 9, device=dev)
        snap_obs = torch.empty(N, env.obs_dim, device=dev); snap_small = torch.empty(N, 9, device=dev)
        gather = (side, g_obs, g_small, snap_obs, snap_small)
    for i in range(W):
        env.step_torch(actions[i])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    done_count = torch.zeros((), device=dev, dtype=torch.int64)
    torch.cuda.synchronize()
    ncu_range = os.environ.get("MW_BENCH_NCU") == "1"     # `ncu --profile-from-start off`: capture the timed region only (launch list under profiles/)
    if ncu_range:
        torch.cuda.profiler.start()
    sampler.begin()
    for i in range(K):
        if not noflush:
            flush.fill_(float(i))                   # evict L2 between timed iterations (outside the event pair)
        ev[i][0].record()
        o, r, te, tr, inf = env.step_torch(actions[W + i])
        if gather is not None:
            # optional epilogue (BASELINE config 4): obs + packed reward/info/flags of every rank to every rank (rank 0 is
            # the learner); copies are taken on the step stream, the two NCCL collectives run on a side stream and
            # overlap the NEXT step's physics
            side, g_obs, g_small, snap_obs, snap_small = gather
            snap_obs.copy_(o); snap_small.copy_(env.d_small)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                dist.all_gather_into_tensor(g_obs, snap_obs); dist.all_gather_into_tensor(g_small, snap_small)
        ev[i][1].record()
        done_count += (te | tr).sum()
    if gather is not None:
        torch.cuda.current_stream(dev).wait_stream(gather[0])
    torch.cuda.synchronize()
    sampler.end()
    if ncu_range:
        torch.cuda.profiler.stop()
    if args.dump_outputs and rank == 0:      # before the profiled pass below overwrites the step buffers
        dump_outputs(args.dump_outputs, dict(obs=o, reward=r, terminated=te, truncated=tr, info=inf))
    if world > 1:
        dist.barrier()
    ms = sum(a.elapsed_time(b) for a, b in ev)
    n_autoreset = int(done_count)
    clocks = sampler.summary()
    sampler.stop_flag = True
    counters = env.engine.counters()
    # ---- profiled pass (not timed): per-phase cycle shares
    env.engine.set_profiling(True)
    env.engine.profile()
    Kp = min(K, 20)
    for i in range(Kp):
        env.step_torch(actions[W + i])
    prof = env.engine.profile()
    env.engine.set_profiling(False)
    t = torch.tensor([ms, e2e_s * 1e3], device=dev, dtype=torch.float64)
    if world > 1 or "MW_BENCH_FAKE_RANK" in os.environ:
        sys.stderr.write(f"[bench] rank {rank} on cuda:{local}: {ms / K:.4f} ms per step (device), e2e {e2e_s * 1e3 / Ke:.4f} ms, "
                         f"own work {(prof['step'] - prof['barrier_wait']) / max(1, N * min(K, 20)):.0f} cycles per env step, "
                         f"convex pairs {prof['n_convex_pairs'] / max(1, N * min(K, 20)):.3f}{' NOFLUSH' if noflush else ''}\n")
    per_rank = None
    if world > 1:
        if dist.get_backend() == "gloo":
            t = t.cpu()
        try:        # every rank's own device time, for the line (the value itself is max-over-ranks, below)
            allt = torch.empty(world * 2, device=t.device, dtype=torch.float64)
            dist.all_gather_into_tensor(allt, t)
            per_rank = [round(float(x) / K, 4) for x in allt.view(world, 2)[:, 0].cpu()]
        except Exception:
            per_rank = None
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, e2e_ms = float(t[0]), float(t[1])
    if rank == 0:
        value = N * world * K / (ms * 1e-3)
        e2e_val = N * world * Ke / (e2e_ms * 1e-3)
        bytes_step = algorithmic_bytes(names)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        achieved = (value / world) * bytes_step / 1e9
        ncu = ncu_summary()
        cpu_val, cpu_sample, flops_step = cpu_baseline(names, 1, args.cpu_steps_per_env, partial=(kind == "ml"))
        obs_dim = env.obs_dim
        own = max(1, prof["step"] - prof["barrier_wait"])
        line = {"metric": METRIC, "value": value, "unit": "env_steps/s", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {"workload": workload_string(args.benchmark, names, n_full, N, kind),
                           "tasks": names, "envs_per_gpu": N,
                           "episode_phase": {"distribution": "uniform 0..499 (permuted over envs)", "min": int(phases.min()), "max": int(phases.max()),
                                             "mean": float(phases.mean()), "autoresets_in_timed_region": n_autoreset,
                                             "expected_autoresets": N * K / 500.0, "pre_roll_steps": 500},
                           "l2": ("NO L2 FLUSH (MW_BENCH_NOFLUSH=1): a diagnosis run, not a benchmark value" if noflush else
                                  "256 MB device write between timed steps (outside the per-step CUDA-event pairs)"),
                           "build": lib().mw_build_info().decode(), "sharding": "env-parallel, no collective on the step path"
                                    + ("; NCCL all_gather_into_tensor of obs + packed reward/info/flags on a side stream (--gather)" if gather else ""),
                           "reference_arm": CPU_ARM_NOTE, "setup_s": round(setup_s, 1), **extra},
                # copies MetaWorldVecEnv.step makes per call: H2D actions [N, 4] f32 (+ the ids of the envs about to truncate, 8 B
                # each); D2H the 39 observation columns the kernel writes (the constant one-hot columns never cross the bus), the
                # packed [N, 9] reward / info / flags record, and the terminal rows (39 + 8 floats) of the finished envs
                "e2e": {"value": e2e_val, "unit": "env_steps/s", "h2d_bytes_per_step": int(N * 4 * 4 + 8 * n_final / max(1, Ke)),
                        "d2h_bytes_per_step": int(N * (39 + 9) * 4 + (39 + 8) * 4 * n_final / max(1, Ke)), "steps": Ke, "autoresets": n_final},
                "gpu_launches": 3 * K,
                **({"per_rank_ms_per_step": per_rank, "per_rank_note": "device time of every rank's own K steps; `ms_per_step` / `value` use the max.  Ranks draw "
                    "their own task-selection / action streams, so the spread is the sample-to-sample spread of the launch's tail "
                    "(profiles/r02_summary.md, Multi-GPU), not communication: the step path has no collective"} if per_rank else {}),
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": ncu.get("dram_bytes_per_launch"), "traffic_source": ncu.get("source"),
                             "algorithmic_bytes_per_launch": bytes_step * N, "algorithmic_bytes_per_env_step": bytes_step,
                             "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650",
                             "flops_per_env_step": flops_step, "achieved_tflops": (value / world) * flops_step / 1e12,
                             "flops_source": "physics flops counted by the float64 oracle (oracle/mjphys.c om_data_flops) on the cpu_baseline sample, resets amortised",
                             "fp32_peak_tflops_nominal": 148 * 128 * 2 * 1.965e9 / 1e12, "ncu": ncu,
                             "note": "latency/issue bound, not HBM bound: one warp runs one env's dependent chain (nv<=17, <1 KB state per env step); "
                                     "the HBM fraction is reported because the metric names it, achieved FLOP/s and active warps are what describe the kernel; see DESIGN.md section 6"},
                "cpu_baseline": {"value": cpu_val, "unit": "env_steps/s", "cores": 1, "kind": "port", "sample": cpu_sample},
                "clocks": clocks,
                "phases": {"unit": "fraction of per-warp own-work cycles (clock64), separate profiled pass of %d steps" % Kp,
                           **{k: round(prof[k] / own, 4) for k in list(prof)[:8]},
                           "barrier_wait_over_own_work": round(prof["barrier_wait"] / own, 4),
                           "warp_cycles_per_env_step_own_work": own / max(1, N * Kp),
                           "convex_pairs_per_env_step": prof["n_convex_pairs"] / max(1, N * Kp),
                           "epa_expansions_per_env_step": prof["n_epa_expansions"] / max(1, N * Kp),
                           "gjk_iters_per_env_step": prof["n_gjk_iters"] / max(1, N * Kp)},
                "solver": {"mean_newton_iters_per_pass": counters["solver_iters"] / max(1, counters["forward_passes"]),
                           "contacts_dropped": counters["contacts_dropped"]}}
        if gather is not None:
            line["gather"] = {"collective": "2 x all_gather_into_tensor per step (obs, packed reward/info/flags), side stream",
                              "bytes_per_rank_per_step": int(N * (obs_dim + 9) * 4), "world": world}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--benchmark", default="MT50", help="MT50 (headline) | MT10 | MT25 | <task>-v3 | ML10-train/test | ML45-train/test")
    ap.add_argument("--envs-per-gpu", type=int, default=4096)
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--e2e-steps", type=int, default=100)
    ap.add_argument("--cpu-steps-per-env", type=int, default=600)
    ap.add_argument("--ref-steps-per-env", type=int, default=1000)
    ap.add_argument("--gather", action="store_true", help="also all-gather obs/reward/flags across ranks every step (BASELINE config 4)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write obs / reward / terminated / truncated / info of the last timed "
                                                          "step (rank 0) as DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0 or args.e2e_steps < 1:
        ap.error("--steps and --e2e-steps must be >= 1 and --warmup >= 0")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
