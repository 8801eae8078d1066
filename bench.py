#!/usr/bin/env python
"""bench.py — learned-dynamics env-steps/sec on N B200s (BASELINE.json metric).

    python bench.py --gpus 1 --steps K --warmup W                 # this repo's CUDA path
    python bench.py --impl reference --gpus 1 --steps K --warmup W  # the reference's CPU algorithm

    python bench.py --config 4 --gpus N ...                        # BASELINE.json configs[3]: 1 M envs + imitation reward
    python bench.py --config 5 --gpus N ...                        # BASELINE.json configs[4]: 8 x (1024 x 4), 512 Ki envs/GPU
    python bench.py ... --dump-outputs DIR                         # also write the last timed step's outputs as DIR/*.npy

One "step" = one pass of the hot path over one batch of synthetic input.  The default workload (--config 2) is
BASELINE.json configs[1], the MILO rollout batch of samples_per_step = 40 000 learned-dynamics env-steps per GPU
with the ensemble discrepancy bonus and the IPM (random-feature) cost — N-member ensemble forward,
s' = s + delta_active, pairwise-max discrepancy, termination mask, cos-feature cost and bonus combine — for the
4 x (512 x 4) dense-connect humanoid3d ensemble (S = 226, A = 28) with random-init weights.  --config 4 adds the
DeepMimic imitation reward (one pose per env) and the global discrepancy quantile over 1 M envs sharded by index;
--config 5 is the 8 x (1024 x 4) ensemble at 512 Ki envs per GPU; --config 3 is the imitation reward alone.

Prints ONE JSON line (rank 0).  `value` is device-resident throughput (inputs already in HBM), `e2e` is the
same work through the host-buffer API with pinned H2D/D2H copies inside the timed region, `roofline` is the
ensemble layer GEMM against the measured tensor peak (burst AND sustained denominators), `sustained` repeats the
timed loop for >= 2 s, `cpu_baseline` is the oracle port of the reference's PyTorch CPU path timed on this box's
host cores on a bounded sample.

--dump-outputs DIR writes what the timed path handed its caller in the last timed step (rank 0's envs): next_state,
disc, done, cost, ipm, bonus and the updated num_steps of the env step, imitation_reward with --config 3 / 4, and with
--config 4 / 5 disc_quantile, the global 0.9 quantile of that step's disc (taken after the timed loop).  Inputs are
seeded, so two builds run with the same arguments can be compared array for array.  See dump_outputs for the format and
the 64 MB cap.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

S_DIM, A_DIM = 226, 28
N_MODELS, HIDDEN = 4, [512, 512, 512, 512]
ENVS_PER_GPU = 40000
RFF_DIM = 512
LAMBDA_B = 0.0025
BW_QUANTILE = 0.1
METRIC = "learned-dynamics env-steps/sec"
UNIT = "env-steps/s"


def flops_per_env_step(n_models=N_MODELS, hidden=HIDDEN, s=S_DIM, a=A_DIM):
    """Algorithmic FLOPs of the ensemble layers (SURVEY.md section 8d): N * 2 * sum_l K_l * O_l."""
    sizes = [s + a] + list(hidden) + [s]
    per_member = sum(2 * sum(sizes[:i + 1]) * sizes[i + 1] for i in range(len(sizes) - 1))
    return n_models * per_member


def fused_bytes_per_env_step(n_models=N_MODELS, s=S_DIM, a=A_DIM):
    """Algorithmic bytes of the fused next-state/discrepancy/termination/cost path (SURVEY.md section 8d)."""
    return s * 4 + a * 4 + n_models * s * 4 + s * 4 + 16 + 1 + 4 + 4


def post_kernel_io_bytes(precision, n_models=N_MODELS, s=S_DIM, rff_k=512, split=True):
    """What post_step_tma_kernel itself moves per env: N member deltas + s in, s' (+ disc, done, counters) out, plus
    the cost features' operand row [hi | lo] of [s; s'] - an implementation artefact, NOT algorithmic bytes."""
    esize = 4 if precision == "tf32" else 2
    return s * 4 * (2 + n_models) + 17 + rff_k * esize * (2 if split else 1)


def profile_note(key):
    """Numbers taken from a committed ncu capture (profiles/roofline_traffic.json), with the run they came from."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if not os.path.exists(p):
        return None, None
    with open(p) as f:
        d = json.load(f)
    return d.get(key), d.get("source")


def hbm_roofline(post_ms, envs, precision, peaks, n_models, split):
    """The step's elementwise tail (next state + discrepancy + termination, the 'reward/cost kernel' of the north
    star) against the measured HBM copy peak, on SURVEY.md section 8(d)'s ALGORITHMIC bytes B_fused(N)."""
    if not post_ms:
        return None
    b = fused_bytes_per_env_step(n_models)
    gbs = b * envs / (post_ms * 1e-3) / 1e9
    io = post_kernel_io_bytes(precision, n_models, split=split)
    traffic, src = profile_note("post_step_dram_bytes_per_launch")
    return {"kernel": "post_step_tma_kernel (next state + discrepancy + termination; also writes the cost operand rows)",
            "bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
            "algorithmic_bytes_per_env_step": b, "kernel_io_bytes_per_env_step": io,
            "achieved_on_kernel_io": io * envs / (post_ms * 1e-3) / 1e9, "traffic": traffic, "traffic_source": src,
            "ms_per_step": post_ms}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm_gbs=d["hbm_gbs"], tensor_tflops=d["bf16_tflops_sustained"], burst_tflops=d["bf16_tflops"],
                    source="measured (MEASURED_PEAKS.json: STREAM copy; bf16 cuBLAS best-of-10 = burst, 4 s loop = sustained)")
    return dict(hbm_gbs=6650.0, tensor_tflops=1400.0, burst_tflops=1590.0, source="fallback (B200_PROFILING.md)")


def tensor_roofline(achieved, timed_seconds, peaks):
    """Both denominators; `frac` is the one that matches the timed region: a region shorter than a second runs at
    burst clocks (nothing has throttled yet), a seconds-long one under the power cap."""
    if not achieved:
        return {"achieved": None, "frac": None}
    burst = timed_seconds < 1.0
    return {"achieved": achieved, "peak": peaks["burst_tflops"] if burst else peaks["tensor_tflops"],
            "frac": achieved / (peaks["burst_tflops"] if burst else peaks["tensor_tflops"]),
            "frac_burst": achieved / peaks["burst_tflops"], "frac_sustained": achieved / peaks["tensor_tflops"],
            "peak_burst": peaks["burst_tflops"], "peak_sustained": peaks["tensor_tflops"],
            "frac_is": "burst" if burst else "sustained", "timed_region_s": timed_seconds}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if t0 <= t <= t1 + 0.15] or [r for (_, r) in self.rows[-3:]]
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except Exception:
                continue
            for name, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def synth_dataset(M, seed):
    import torch
    g = torch.Generator().manual_seed(seed)
    s = torch.randn(M, S_DIM, generator=g)
    a = torch.randn(M, A_DIM, generator=g)
    return s, a, s + 0.05 * torch.randn(M, S_DIM, generator=g)


def synth_expert(M, seed):
    import torch
    g = torch.Generator().manual_seed(seed)
    es = torch.randn(M, S_DIM, generator=g)
    return torch.cat([es, es + 0.05 * torch.randn(M, S_DIM, generator=g)], dim=1)


# ======================================================================================================
# workloads (BASELINE.json configs, 1-based as the verdict numbers them)

CONFIGS = {
    2: dict(n_models=4, hidden=[512] * 4, envs_per_gpu=40000, envs_total=None, imitation=False, quantile_every=0,
            scaling="weak", name="configs[1]: MILO rollout batch, 40 000 learned-dynamics env-steps per GPU per step with "
                                 "ensemble discrepancy bonus + IPM/RFF cost"),
    3: dict(n_models=4, hidden=[512] * 4, envs_per_gpu=None, envs_total=1 << 20, imitation=True, quantile_every=0,
            scaling="strong", name="configs[2]: DeepMimic/AMP imitation reward only, 1 M synthetic humanoid3d poses vs the "
                                   "spinkick clip"),
    4: dict(n_models=4, hidden=[512] * 4, envs_per_gpu=None, envs_total=1 << 20, imitation=True, quantile_every=10,
            scaling="strong", name="configs[3]: fused ensemble step + discrepancy quantile + MILO cost + imitation reward, "
                                   "1 M parallel envs sharded by index"),
    5: dict(n_models=8, hidden=[1024] * 4, envs_per_gpu=1 << 19, envs_total=None, imitation=False, quantile_every=10,
            scaling="weak", name="configs[4]: 8-model ensemble (hidden 1024 x 4), 512 Ki envs per GPU (4 M at 8 GPUs), global "
                                 "discrepancy quantile via NCCL"),
}


def workload_config(cfg_id, n_gpus, envs_per_gpu, extra=None):
    c = CONFIGS[cfg_id]
    cfg = {
        "workload": c["name"] + f" (BASELINE.json, --config {cfg_id})",
        "ensemble": f"{c['n_models']} x ({c['hidden'][0]} x {len(c['hidden'])}) dense_connect, transform, humanoid3d "
                    f"S=226 A=28, random init base_seed=100",
        "envs_per_gpu": envs_per_gpu, "global_envs_per_step": envs_per_gpu * n_gpus,
        "rff": {"feature_dim": RFF_DIM, "input_type": "ss", "lambda_b": LAMBDA_B},
        "sharding": f"envs by index over {n_gpus} GPU(s), full ensemble replica per GPU",
        "l2_policy": "inputs rotate through a ring of batches larger than the 126 MB L2; activations never fit",
    }
    if extra:
        cfg.update(extra)
    return cfg


# ======================================================================================================
# reference arm: the reference's own CPU algorithm (oracle port of its PyTorch path)


def cpu_reference_setup(n_models, hidden):
    import torch
    from oracle import milo_oracle as mo
    ws, bs = mo.init_ensemble(S_DIM, A_DIM, hidden, n_models, dense_connect=True, base_seed=100)
    ds = synth_dataset(8192, 0)
    tf = mo.get_transformations(*ds)
    cost = mo.RffCostOracle(synth_expert(4096, 2), feature_dim=RFF_DIM, input_type="ss", bw_quantile=BW_QUANTILE,
                            lambda_b=LAMBDA_B, seed=100)
    thr = mo.compute_threshold(ws, bs, tf, ds[0][:1024], ds[1][:1024])
    g = torch.Generator().manual_seed(1)
    cost.w = torch.randn(RFF_DIM, generator=g) * 0.01
    return mo, ws, bs, tf, cost, thr


def cpu_reference_step(ctx, s, a, member, steps):
    """One batch of env-steps as the reference computes them (BASELINE.md section 4.4): active-member
    forward (sim_env.py:155-158), is_done (sim_env.py:164-173), get_bonus_costs = N-member discrepancy +
    RFF cost + combine (linear_cost.py:111-152)."""
    import torch
    mo, ws, bs, tf, cost, thr = ctx
    with torch.no_grad():
        nxt = torch.empty_like(s)
        for m in range(len(ws)):  # the reference steps each env with its own active member
            idx = (member == m).nonzero(as_tuple=False).squeeze(1)
            if idx.numel():
                nxt[idx] = s[idx] + mo.dynamics_forward(ws[m], bs[m], tf, s[idx], a[idx])
        _, st, done = mo.simenv_step(s.double().numpy(), (nxt - s).numpy(), steps.numpy())
        disc = mo.compute_discrepancy(ws, bs, tf, s, a)
        c, _ = cost.get_bonus_costs(s, a, disc, thr, next_states=nxt)
    return nxt, c, done


def cpu_imitation_rate(seconds=4.0):
    """poses/s of the reference's own compiled reward code (oracle/_ref/libdmref.so, built from the reference's
    sources by oracle/ref_build.py) on one host core; None when the checker library was not shipped."""
    try:
        import ctypes
        import numpy as np
        from oracle import ref_build
        lib = ref_build.load()
        if lib is None:
            return None
        n, dof = 1024, lib.dmref_num_dof()
        PD = ctypes.POINTER(ctypes.c_double)
        rng = np.random.default_rng(3)
        tt = np.ascontiguousarray(rng.uniform(0.0, lib.dmref_duration(), size=n))
        pp, vv = np.zeros((n, dof)), np.zeros((n, dof))
        tmp_t = np.zeros(1)
        for i in range(n):  # pose = clip(t) perturbed (SURVEY.md section 8d)
            lib.dmref_kin_pose_vel(tt[i], None, pp[i].ctypes.data_as(PD), vv[i].ctypes.data_as(PD))
        pp[:, :3] += 0.05 * rng.standard_normal((n, 3))
        vv += 0.5 * rng.standard_normal(vv.shape)
        out = np.zeros(n)
        call = lambda: lib.dmref_reward_batch(n, pp.ctypes.data_as(PD), vv.ctypes.data_as(PD), tt.ctypes.data_as(PD),  # noqa: E731
                                              None, out.ctypes.data_as(PD), None)
        call()
        t0, reps = time.perf_counter(), 0
        while time.perf_counter() - t0 < seconds:
            call()
            reps += 1
        return n * reps / (time.perf_counter() - t0)
    except Exception:
        return None


def time_cpu_reference(cfg_id, batch, min_seconds, max_reps, warmup=1):
    import torch
    c = CONFIGS[cfg_id]
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    ctx = cpu_reference_setup(c["n_models"], c["hidden"])
    g = torch.Generator().manual_seed(1)
    s, a = torch.randn(batch, S_DIM, generator=g), torch.randn(batch, A_DIM, generator=g)
    member = torch.randint(0, c["n_models"], (batch,), generator=g)
    steps = torch.zeros(batch, dtype=torch.int64)
    for _ in range(warmup):
        cpu_reference_step(ctx, s, a, member, steps)
    times = []
    t_start = time.perf_counter()
    while len(times) < max_reps and (time.perf_counter() - t_start < min_seconds or len(times) < 3):
        t0 = time.perf_counter()
        cpu_reference_step(ctx, s, a, member, steps)
        times.append(time.perf_counter() - t0)
    med = statistics.median(times)
    # the reference's ACTUAL mode steps one env per call (sim_env.py:155-157 unsqueezes a single state); reported
    # beside the batched figure, which is the generous one (SURVEY.md section 8d)
    one = []
    for i in range(60):
        t0 = time.perf_counter()
        cpu_reference_step(ctx, s[i:i + 1], a[i:i + 1], member[i:i + 1], steps[i:i + 1])
        one.append(time.perf_counter() - t0)
    return dict(value=batch / med, unit=UNIT, cores=threads, kind="port",
                sample=f"{len(times)} x {batch} env-steps (median; a SAMPLE of the GPU arm's batch, rate per env-step), "
                       f"oracle port of the reference's PyTorch CPU path, torch {torch.__version__} with {threads} "
                       f"intra-op threads",
                per_env_mode={"value": 1.0 / statistics.median(one[10:]), "unit": UNIT,
                              "sample": "50 single-env steps (median): the batch the reference's SimEnv.step uses"}), med


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (oracle port; the reference itself is Python and cannot
    travel to the GPU box) on all host threads.  Each step is a bounded SAMPLE of the GPU arm's batch (the rate is
    per env-step, so the sample size does not bias it), sized after one probe step so that the whole run stays within
    a couple of minutes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import torch
    c = CONFIGS[args.config]
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    ctx = cpu_reference_setup(c["n_models"], c["hidden"])
    g = torch.Generator().manual_seed(1)
    full = 4096
    s, a = torch.randn(full, S_DIM, generator=g), torch.randn(full, A_DIM, generator=g)
    member = torch.randint(0, c["n_models"], (full,), generator=g)
    steps = torch.zeros(full, dtype=torch.int64)
    cpu_reference_step(ctx, s[:256], a[:256], member[:256], steps[:256])
    t0 = time.perf_counter()
    cpu_reference_step(ctx, s, a, member, steps)
    probe = time.perf_counter() - t0
    budget = 100.0 / max(args.steps + args.warmup, 1)  # seconds per step
    batch = int(max(256, min(full, (full * budget / probe) // 256 * 256)))
    s, a, member, steps = s[:batch], a[:batch], member[:batch], steps[:batch]
    for _ in range(max(args.warmup, 1)):
        cpu_reference_step(ctx, s, a, member, steps)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_reference_step(ctx, s, a, member, steps)
    dt = time.perf_counter() - t0
    value = batch * args.steps / dt
    envs_per_gpu = c["envs_per_gpu"] or c["envs_total"] // max(args.gpus, 1)
    sample = (f"each step = {batch} env-steps, a sample of the {envs_per_gpu}-step batch of the GPU arm (rate per "
              f"env-step), oracle port of the reference's PyTorch CPU path, torch {torch.__version__}, {threads} "
              f"intra-op threads")
    extra = {"cpu_sample": sample}
    if c["imitation"]:
        r = cpu_imitation_rate()
        if r:
            extra["cpu_imitation_poses_per_s_one_core"] = r
            value = 1.0 / (1.0 / value + 1.0 / (r * threads))  # step + one reward per env, reward on every core
            sample += f"; + the compiled reference reward code at {r:.0f} poses/s/core x {threads} cores"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": c["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.config, args.gpus, envs_per_gpu, extra=extra),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


# ======================================================================================================
# this repo's arm


class RolloutStats:
    """Rollout cost / discrepancy statistics (batch_reinforce.py:135-141) kept OFF the compute stream: every step's
    [max, sum] of cost and discrepancy is reduced on a side stream behind an event, into one row of a device block;
    every `every` steps that block crosses NCCL once (all-gather of every x 4 doubles).  Runs at every world size, so
    the compute stream is identical at 1 and at 8 GPUs."""

    def __init__(self, eng, device, world, every=10, ring=4):
        import torch
        self.torch, self.eng, self.world, self.every = torch, eng, world, every
        self.side = torch.cuda.Stream(device)
        self.rows = torch.zeros((every, 4), device=device, dtype=torch.float64)
        self.gathered = torch.zeros((world * every * 4,), device=device, dtype=torch.float64)
        self.k = 0
        self.collectives = 0
        self.free = [None] * ring  # side-stream event per output slot: the slot may be overwritten after it

    def before_step(self, slot):
        if self.free[slot] is not None:
            self.torch.cuda.current_stream().wait_event(self.free[slot])

    def after_step(self, slot, cst, disc):
        torch = self.torch
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream())
        with torch.cuda.stream(self.side):
            self.side.wait_event(ev)
            self.eng.reduce_max_sum(cst, out=self.rows[self.k, 0:2])
            self.eng.reduce_max_sum(disc, out=self.rows[self.k, 2:4])
            done = torch.cuda.Event()
            done.record(self.side)
            self.free[slot] = done
            self.k += 1
            if self.k == self.every:
                self.k = 0
                if self.world > 1:
                    import torch.distributed as dist
                    dist.all_gather_into_tensor(self.gathered, self.rows.view(-1))
                    self.collectives += 1

    def join(self):
        self.torch.cuda.current_stream().wait_stream(self.side)


def pcie_probe(device, nbytes=36 << 20, reps=10):
    """GB/s of back-to-back pinned device->host copies of one step's result size, all ranks at once: what the box's
    PCIe gives a rank while its neighbours copy too."""
    import torch
    d = torch.empty(nbytes, device=device, dtype=torch.uint8)
    h = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    for _ in range(2):
        h.copy_(d, non_blocking=True)
    torch.cuda.synchronize(device)
    t0 = time.perf_counter()
    for _ in range(reps):
        h.copy_(d, non_blocking=True)
    torch.cuda.synchronize(device)
    return nbytes * reps / (time.perf_counter() - t0) / 1e9


DUMP_LIMIT_BYTES = 64_000_000


def dump_outputs(out_dir, per_env, scalars=None, limit=DUMP_LIMIT_BYTES):
    """Writes per_env's tensors (first dimension = env) as out_dir/<name>.npy: floating outputs as float32, integer
    ones (done, num_steps) as float64.  When they exceed `limit` bytes together, every array keeps the same rows, a
    sorted sample drawn with a fixed seed, and rows.npy holds their indices.  scalars are written as 1-element float64
    arrays."""
    import numpy as np
    import torch
    n = next(iter(per_env.values())).shape[0]
    row_bytes = sum((t[0].numel() if t.dim() > 1 else 1) * (4 if t.is_floating_point() else 8) for t in per_env.values())
    os.makedirs(out_dir, exist_ok=True)
    rows = None
    if n * row_bytes > limit:
        keep = (limit - 65536) // (row_bytes + 8)   # rows.npy and the .npy headers fit in the 64 KiB kept back
        rows = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:keep].sort().values
        np.save(os.path.join(out_dir, "rows.npy"), rows.numpy().astype(np.float64))
    for name, t in per_env.items():
        t = t.detach() if rows is None else t.detach()[rows.to(t.device)]
        t = t.float() if t.is_floating_point() else t.double()
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())
    for name, v in (scalars or {}).items():
        np.save(os.path.join(out_dir, name + ".npy"), np.array([v], dtype=np.float64))


def run_ours(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    from amp_extensions_b200 import AmpDataset, DynamicsEnsemble, ImitationReward, RBFLinearCost, _lib
    from amp_extensions_b200.engine import HumanoidTermination
    from amp_extensions_b200.host_api import HostEnvPipeline, HostStepPipeline
    from amp_extensions_b200 import parallel
    host_cpus = parallel.bind_host_to_gpu(local_rank)  # NUMA-local pinned buffers for the host-buffer pass

    C = CONFIGS[args.config]
    n_models, hidden = C["n_models"], C["hidden"]
    if C["envs_total"] is not None and args.envs is None:
        lo, hi = parallel.shard_range(C["envs_total"], rank, world)
        E = hi - lo
    else:
        E = args.envs if args.envs is not None else C["envs_per_gpu"]
    step_on = args.config != 3
    ds = AmpDataset(*synth_dataset(8192, 0))
    ens = DynamicsEnsemble(S_DIM, A_DIM, ds, None, num_models=n_models, hidden_sizes=hidden, dense_connect=True,
                           transform=True, base_seed=100, precision=args.precision, device=device)
    eng = ens.engine()
    eng.set_termination(HumanoidTermination(horizon=300))
    cost = RBFLinearCost(synth_expert(4096, 2), feature_dim=RFF_DIM, input_type="ss", bw_quantile=BW_QUANTILE,
                         lambda_b=LAMBDA_B, seed=100, precision=args.precision, device=device)
    eng.load_rff(cost.rff.weight.data, cost.rff.bias.data, split=True)
    # discrepancy threshold: dataset maximum, global over ranks (dynamics.py:145-152)
    ens.train_dataset = AmpDataset(ds.states[rank::world][:1024], ds.actions[rank::world][:1024],
                                   ds.next_states[rank::world][:1024])
    threshold = parallel.global_threshold(ens)

    # input ring larger than L2 (126 MB): E * 1016 B per batch
    ring = max(2, min(8, -(-(160 << 20) // (E * (S_DIM + A_DIM) * 4))))
    oring = 4  # per-step output rows (the rollout's time-major buffers): the statistics side stream reads them
    g = torch.Generator(device=device).manual_seed(1 + rank)
    states = [torch.randn(E, S_DIM, device=device, generator=g) for _ in range(ring)]
    actions = [torch.randn(E, A_DIM, device=device, generator=g) for _ in range(ring)]
    member = torch.randint(0, n_models, (E,), device=device, generator=g, dtype=torch.int32)
    steps = torch.zeros(E, device=device, dtype=torch.int32)
    nxt = torch.empty(E, S_DIM, device=device)
    disc, cst = (torch.empty(oring, E, device=device) for _ in range(2))
    ipm, bonus = (torch.empty(E, device=device) for _ in range(2))
    done = torch.empty(E, device=device, dtype=torch.uint8)
    # cost weights: fit on the first 1024 rollout rows (batch_reinforce.py:113), global mean over ranks
    n_fit = min(E, 1024)
    eng.step(states[0][:n_fit], actions[0][:n_fit], member[:n_fit], steps[:n_fit].clone(), next_state=nxt[:n_fit],
             disc=disc[0][:n_fit], done=done[:n_fit])
    w = parallel.global_fit_cost(cost, torch.cat([states[0][:n_fit], nxt[:n_fit]], dim=1)).to(device)
    # hi/lo operand pairs of the cost-feature GEMM only where plain operands measurably miss the budget
    split_report = cost.split_decision(torch.cat([states[0][:384], nxt[:384]], dim=1).cpu(), w.cpu())
    use_split = {"auto": split_report["split"], "on": True, "off": False}[args.rff_split]
    eng.set_rff_split(use_split)
    split_report["used"] = bool(use_split)

    imit, poses = None, None
    if C["imitation"]:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        from bench_imitation import synth_poses
        imit = ImitationReward(device=device)
        poses = [synth_poses(imit, E, device, seed=3 + 7 * rank + i) for i in range(2)]
        rew = torch.empty(E, device=device)
    stats = RolloutStats(eng, device, world, every=10, ring=oring)
    q_every = C["quantile_every"]
    q_state = {"value": None, "calls": 0, "wall_s": 0.0, "events": []}

    def one_step(i):
        k, o = i % ring, i % oring
        if step_on:
            stats.before_step(o)
            eng.step_cost(states[k], actions[k], member, steps, w, LAMBDA_B, threshold, next_state=nxt, disc=disc[o],
                          done=done, cost=cst[o], ipm=ipm, bonus=bonus)
            stats.after_step(o, cst[o], disc[o])
        if imit is not None:
            p, v, t = poses[i % 2]
            imit.reward(p, v, t, out=rew)
        if q_every and (i + 1) % q_every == 0:
            t0 = time.perf_counter()
            qe0, qe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            qe0.record()
            q_state["value"] = parallel.global_quantile(disc[o], 0.9, engine=eng)  # one host sync, inside the region
            qe1.record()
            q_state["events"].append((qe0, qe1))
            q_state["wall_s"] += time.perf_counter() - t0   # includes draining the steps queued ahead of the sync
            q_state["calls"] += 1

    def barrier():
        torch.cuda.synchronize(device)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    # ---- multi-GPU parity: every rank's shard equals rank 0's recomputation of the same rows, bit for bit -------
    shard_parity = None
    if world > 1 and step_on:
        P = 1024
        gp = torch.Generator(device=device).manual_seed(999)  # same stream on every rank
        ps = torch.randn(world * P, S_DIM, device=device, generator=gp)
        pa = torch.randn(world * P, A_DIM, device=device, generator=gp)
        pm = torch.randint(0, n_models, (world * P,), device=device, generator=gp, dtype=torch.int32)

        def run_rows(r0, r1):
            o_n = torch.empty(r1 - r0, S_DIM, device=device)
            o_d, o_c, o_i, o_b = (torch.empty(r1 - r0, device=device) for _ in range(4))
            o_f = torch.empty(r1 - r0, device=device, dtype=torch.uint8)
            eng.step_cost(ps[r0:r1].contiguous(), pa[r0:r1].contiguous(), pm[r0:r1].contiguous(),
                          torch.zeros(r1 - r0, device=device, dtype=torch.int32), w, LAMBDA_B, threshold, next_state=o_n,
                          disc=o_d, done=o_f, cost=o_c, ipm=o_i, bonus=o_b)
            return torch.cat([o_n, o_d[:, None], o_c[:, None], o_f[:, None].float()], dim=1)

        mine = run_rows(rank * P, (rank + 1) * P)
        allr = torch.empty(world * P, mine.shape[1], device=device)
        dist.all_gather_into_tensor(allr, mine)
        ok = torch.ones(1, device=device)
        if rank == 0:
            whole = run_rows(0, world * P)  # one call over every rank's rows (chunk boundaries differ too)
            ok[0] = 1.0 if torch.equal(whole, allr) else 0.0
        dist.broadcast(ok, 0)
        if ok.item() != 1.0:
            raise SystemExit("shard parity FAILED: a rank's rows differ from rank 0's recomputation")
        shard_parity = "ok"

    def timed(n_steps, first):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n_steps):
            one_step(first + i)
        stats.join()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    for i in range(args.warmup):
        one_step(i)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = _lib.launch_count()
    t_wall0 = time.time()
    total_ms = timed(args.steps, args.warmup)
    t_wall1 = time.time()
    launches = _lib.launch_count() - launches0
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    if args.dump_outputs:   # now: the passes below write into the same output buffers
        o = (args.warmup + args.steps - 1) % oring
        scalars = {}
        if q_every and step_on:   # a collective: every rank takes part
            scalars["disc_quantile"] = float(parallel.global_quantile(disc[o], 0.9, engine=eng))
        if rank == 0:
            per_env = {}
            if step_on:
                per_env.update(next_state=nxt, disc=disc[o], done=done, cost=cst[o], ipm=ipm, bonus=bonus,
                               num_steps=steps)
            if imit is not None:
                per_env["imitation_reward"] = rew
            dump_outputs(args.dump_outputs, per_env, scalars)
    e_total = torch.tensor([float(E)], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e_total, op=dist.ReduceOp.SUM)
    envs_global = float(e_total.item())
    value = envs_global * args.steps / (total_ms * 1e-3)
    torch.cuda.synchronize(device)
    quantile = {"value": q_state["value"], "calls": q_state["calls"],
                "device_ms_per_call": (sum(a.elapsed_time(b) for a, b in q_state["events"]) / len(q_state["events"]))
                if q_state["events"] else None,
                "host_wall_ms_per_call": (q_state["wall_s"] / q_state["calls"] * 1e3) if q_state["calls"] else None,
                "note": "device = the quantile's own launches and collectives (CUDA events); host wall also counts the "
                        "queued steps the call's single synchronisation has to drain"}
    q_state.update(calls=0, wall_s=0.0, events=[])

    # ---- sustained: the same loop for >= 2 s, with its own clock record ---------------------------------------
    sustained = None
    if not args.skip_sustained:
        n_sus = max(args.steps, int(2200.0 / max(total_ms / args.steps, 1e-3)))
        s2 = ClockSampler(local_rank)
        if rank == 0:
            s2.start()
        tw0 = time.time()
        sus_ms = timed(n_sus, 0)
        tw1 = time.time()
        sustained = {"value": envs_global * n_sus / (sus_ms * 1e-3), "unit": UNIT, "steps": n_sus,
                     "ms_per_step": sus_ms / n_sus, "seconds": sus_ms * 1e-3,
                     "clocks": s2.stop(tw0, tw1) if rank == 0 else None}
        q_state.update(calls=0, wall_s=0.0, events=[])

    # ---- diagnostic: the same steps replayed from CUDA graphs (no per-launch CPU work at all) ------------
    graph_ms = None
    if args.graph_check and world == 1 and not q_every:
        graphs = []
        for k in range(ring):
            gk = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gk):
                eng.step_cost(states[k], actions[k], member, steps, w, LAMBDA_B, threshold, next_state=nxt, disc=disc[0],
                              done=done, cost=cst[0], ipm=ipm, bonus=bonus)
            graphs.append(gk)
        for i in range(args.warmup):
            graphs[i % ring].replay()
        torch.cuda.synchronize(device)
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for i in range(args.steps):
            graphs[i % ring].replay()
        g1.record()
        torch.cuda.synchronize(device)
        graph_ms = g0.elapsed_time(g1) / args.steps

    # ---- per-kernel device time (CUDA events inside the library, same workload, separate pass) ----------
    prof_steps = max(3, min(args.steps, 50 if E <= 65536 else 5))
    per_step = {}
    if step_on:
        eng.profile_enable(True)
        for i in range(prof_steps):
            eng.step_cost(states[i % ring], actions[i % ring], member, steps, w, LAMBDA_B, threshold, next_state=nxt,
                          disc=disc[0], done=done, cost=cst[0], ipm=ipm, bonus=bonus)
        prof = eng.profile_read(reset=True)
        eng.profile_enable(False)
        per_step = {k: v[0] / prof_steps for k, v in prof.items() if v[1] > 0}
    imit_ms = None
    if imit is not None:
        n_im = 30
        for i in range(3):
            imit.reward(*poses[i % 2], out=rew)
        torch.cuda.synchronize(device)
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for i in range(n_im):
            p, v, t = poses[i % 2]
            imit.reward(p, v, t, out=rew)
        a1.record()
        torch.cuda.synchronize(device)
        imit_ms = a0.elapsed_time(a1) / n_im
        per_step["imitation"] = imit_ms

    if args.skip_e2e:
        if rank == 0:
            emit({"metric": METRIC, "value": value, "unit": UNIT, "ms_per_step": total_ms / args.steps,
                  "kernels_ms_per_step": per_step, "rff_split": split_report,
                  "note": "profiling run (--skip-e2e), not a bench line"})
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- end to end through the host-buffer API: pinned H2D + step + D2H inside the timed region ----------
    e2e = None
    if step_on:
        nhs = 2
        hs = [states[k].cpu().pin_memory() for k in range(nhs)]
        ha = [actions[k % ring].cpu().pin_memory() for k in range(4)]
        hm, hst = member.cpu().pin_memory(), torch.zeros(E, dtype=torch.int32).pin_memory()
        e2e_steps = max(6, min(args.steps, 100 if E <= 65536 else 6))
        chunks = args.e2e_chunks if E <= 65536 else max(args.e2e_chunks, -(-E // 65536))
        hp, hv, ht = (None, None, None)
        if imit is not None:
            hp, hv, ht = (x.cpu().pin_memory() for x in poses[0])
            dp, dv, dt_ = (torch.empty_like(x) for x in poses[0])
            h_rew = torch.empty(E, dtype=torch.float32, pin_memory=True)

        def timed_host_loop(submit, collect):
            """Two groups of envs alternate: group i+1's upload and group i-1's download overlap group i's compute.
            Every step's inputs cross PCIe host->device and every step's results (next state, cost, done, disc,
            counters; the imitation reward in config 4) come back and are read on the host."""
            for i in range(8):
                submit(i)
                collect()
            barrier()
            t0 = time.perf_counter()
            chk = 0.0
            submit(0)
            for i in range(1, e2e_steps):
                submit(i)
                out = collect()
                chk += float(out[-1]["cost"][0]) + float(out[0]["next"][-1, -1])  # the caller reads the results
            out = collect()
            chk += float(out[-1]["cost"][0]) + float(out[0]["next"][-1, -1])
            torch.cuda.synchronize(device)
            dt = torch.tensor([time.perf_counter() - t0], device=device, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            return envs_global * e2e_steps / float(dt.item())

        # (1) the plugin's own call shape, env.step(actions): state resident on the device (sim_env.py:140-162)
        envp = HostEnvPipeline(eng, E, groups=2, n_chunks=chunks, with_cost=True)
        envp.reset(0, hs[0], hm)
        envp.reset(1, hs[1], hm)
        extra_h2d = extra_d2h = 0

        def submit_env(i):
            envp.submit(i % 2, ha[i % 4], w, LAMBDA_B, threshold)
            if imit is not None:  # the simulated character's pose / velocity come from the caller in this path
                dp.copy_(hp, non_blocking=True); dv.copy_(hv, non_blocking=True); dt_.copy_(ht, non_blocking=True)
                imit.reward(dp, dv, dt_, out=rew)
                h_rew.copy_(rew, non_blocking=True)

        if imit is not None:
            extra_h2d = E * (43 + 43 + 1) * 4
            extra_d2h = E * 4
        e2e_value = timed_host_loop(submit_env, envp.collect_chunks)
        e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": envp.h2d_bytes_per_step + extra_h2d,
               "d2h_bytes_per_step": envp.d2h_bytes_per_step + extra_d2h, "steps": e2e_steps, "chunks": len(envp.bounds),
               "api": "amp_extensions_b200.host_api.HostEnvPipeline.submit/collect_chunks: env.step(actions) on pinned "
                      "host actions, env state resident on the device as in SimEnv (sim_env.py:140-162); obs / cost / "
                      "done / disc / counters come back as ONE packed record per chunk and are read on the host; 2 env "
                      "groups alternate",
               "host_cpus_rank0": (f"{len(host_cpus)} cores near the GPU (NVML affinity)" if host_cpus else "unbound")}
        # the same without the optional blocks (a sampler that needs obs / cost / done only)
        lean = HostEnvPipeline(eng, E, groups=2, n_chunks=chunks, with_cost=True, want_disc=False, want_steps=False)
        lean.reset(0, hs[0], hm)
        lean.reset(1, hs[1], hm)
        e2e["lean"] = {"value": timed_host_loop(lambda i: lean.submit(i % 2, ha[i % 4], w, LAMBDA_B, threshold),
                                                lean.collect_chunks),
                       "d2h_bytes_per_step": lean.d2h_bytes_per_step, "what": "obs + cost + done only"}
        del lean
        # half-precision observations (opt-in): half the bytes per step where the host's PCIe is the limit
        half = HostEnvPipeline(eng, E, groups=2, n_chunks=chunks, with_cost=True, want_disc=False, want_steps=False,
                               obs_dtype=torch.float16)
        half.reset(0, hs[0], hm)
        half.reset(1, hs[1], hm)
        e2e["obs_fp16"] = {"value": timed_host_loop(lambda i: half.submit(i % 2, ha[i % 4], w, LAMBDA_B, threshold),
                                                    half.collect_chunks),
                           "d2h_bytes_per_step": half.d2h_bytes_per_step,
                           "what": "obs (fp16, 2^-11 relative rounding) + cost + done; the state stays fp32 on the device"}
        del half
        # (2) stateless callers: the full state crosses PCIe both ways every step
        if E <= 65536:
            pipe = HostStepPipeline(eng, E, n_chunks=chunks, with_cost=True)

            def collect_stateless():
                o = pipe.collect()
                return [{"next": o[0], "cost": o[1]}]

            e2e["stateless"] = {
                "value": timed_host_loop(lambda i: pipe.submit(hs[i % nhs], ha[i % 4], hm, hst, w, LAMBDA_B, threshold),
                                         collect_stateless),
                "h2d_bytes_per_step": pipe.h2d_bytes_per_step, "d2h_bytes_per_step": pipe.d2h_bytes_per_step,
                "api": "HostStepPipeline.submit/collect: full state uploaded every step"}
            del pipe
        # what the box's PCIe can do for one step's results, every rank at once (the e2e ceiling at N > 1)
        barrier()
        gbs = torch.tensor([pcie_probe(device, nbytes=min(max(envp.d2h_bytes_per_step, 1 << 20), 256 << 20))],
                           device=device, dtype=torch.float64)
        if world > 1:
            allg = torch.empty(world, device=device, dtype=torch.float64)
            dist.all_gather_into_tensor(allg, gbs)
            gbs = allg
        e2e["pcie_d2h_probe_gbs_per_rank"] = [round(float(x), 2) for x in gbs.tolist()]
        e2e["pcie_probe_implied_env_steps_per_s"] = float(gbs.min()) * 1e9 / (envp.d2h_bytes_per_step / E) * world
        del envp

    # ---- device-resident policy: the supported large-scale calling mode (no per-step PCIe at all) ------------
    device_policy = None
    if args.config == 2 and not args.skip_extras:
        try:
            device_policy = device_policy_rollout(ens, cost, ds, E, device, world, barrier)
        except Exception as ex:  # report, do not hide
            device_policy = {"error": repr(ex)[:300]}
    single_env = None
    if args.config == 2 and rank == 0 and not args.skip_extras:
        try:
            single_env = plugin_single_env(ens, ds, device)
        except Exception as ex:
            single_env = {"error": repr(ex)[:300]}

    if rank == 0:
        peaks = measured_peaks()
        gemm_ms = per_step.get("ensemble_gemm")
        flop = flops_per_env_step(n_models, hidden)
        achieved = flop * E / (gemm_ms * 1e-3) / 1e12 if gemm_ms else None
        traffic, tsrc = profile_note("ensemble_gemm_dram_bytes_per_step") if args.config == 2 else (None, None)
        cpu = None
        if not args.skip_cpu_baseline:
            cpu, _ = time_cpu_reference(args.config, 1024 if n_models <= 4 else 512, min_seconds=12.0, max_reps=200)
            if single_env and "value" in single_env:
                cpu["per_env_mode"]["gpu_plugin_single_env"] = single_env
        fwd = eng.forward_launches(E)
        roof = {"kernel": ("ensemble_chain_kernel (all ensemble layers of a (member, 256-row env tile) on one CTA pair, "
                           "one launch per chunk)" if fwd == 1 else
                           f"gemm_tcgen05_kernel ({fwd} ensemble layer launches per chunk)"), "bound": "tensor",
                "unit": "TFLOP/s", "traffic": traffic, "traffic_source": tsrc, "peak_source": peaks["source"],
                "algorithmic_flop_per_env_step": flop, "ms_per_step": gemm_ms}
        roof.update(tensor_roofline(achieved, total_ms * 1e-3, peaks))
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": C["scaling"], "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
            "config": workload_config(args.config, world, E, extra={
                "operands": f"{args.precision} in, fp32 accumulate (TMEM)", "threshold": threshold,
                "rff_split": split_report,
                "statistics": f"per-step [max, sum] of cost and discrepancy on a side stream, one all-gather per 10 steps "
                              f"({stats.collectives} collectives in all timed loops)"}),
            "clocks": clocks, "e2e": e2e, "sustained": sustained, "gpu_launches": int(launches),
            "roofline": roof, "kernels_ms_per_step": per_step, "graph_replay_ms_per_step": graph_ms,
            "roofline_hbm": hbm_roofline(per_step.get("post"), E, args.precision, peaks, n_models, use_split),
            "cpu_baseline": cpu, "shard_parity": shard_parity,
        }
        if q_every:
            line["quantile"] = quantile
        if imit_ms:
            gbs_i = 352 * E / (imit_ms * 1e-3) / 1e9
            fl, fsrc = profile_note("imitation_fp32_pipe_frac")
            line["roofline_imitation"] = {
                "kernel": "imitation_reward_h3d_kernel", "bound": "hbm", "achieved": gbs_i, "peak": peaks["hbm_gbs"],
                "unit": "GB/s", "frac": gbs_i / peaks["hbm_gbs"], "algorithmic_bytes_per_pose": 352,
                "ms_per_step": imit_ms, "fp32_pipe_frac": fl, "fp32_pipe_frac_source": fsrc}
        if device_policy is not None:
            line["e2e_device_policy"] = device_policy
        if single_env is not None:
            line["plugin_single_env"] = single_env
        if args.config == 3:
            line["metric"], line["unit"] = "imitation-reward poses/sec", "poses/s"
            line["note"] = "configs[2] is a parity / kernel configuration, not the headline metric"
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


class _FC:
    """mjrl FCNetwork stand-in (fc_network.py:42-55): 226 -> 32 -> 32 -> 28 tanh, run.py's policy_size."""

    def __init__(self, sizes, seed):
        import torch
        g = torch.Generator().manual_seed(seed)
        self.fc_layers = [torch.nn.Linear(sizes[i], sizes[i + 1]) for i in range(len(sizes) - 1)]
        for l in self.fc_layers:
            l.weight.data = torch.randn(l.weight.shape, generator=g) * (1.0 / l.weight.shape[1]) ** 0.5
            l.bias.data = torch.zeros(l.bias.shape)
        self.fc_layers[-1].weight.data *= 1e-2   # gaussian_mlp.py:38-39
        self.nonlinearity = torch.tanh
        self.in_shift, self.in_scale = torch.zeros(sizes[0]), torch.ones(sizes[0])
        self.out_shift, self.out_scale = torch.zeros(sizes[-1]), torch.ones(sizes[-1])


class _Policy:
    def __init__(self, obs, act, seed=123):
        import torch
        self.model = _FC((obs, 32, 32, act), seed)
        self.log_std = torch.full((act,), -0.5)


def device_policy_rollout(ens, cost, ds, E, device, world, barrier, horizon=32, iters=6):
    """env-steps/s of rollout.DeviceRollout.collect: Gaussian MLP policy + env step + cost + auto-reset on the device
    over a 32-step horizon, the whole batch of paths downloaded to pinned host memory ONCE per horizon (inside the
    timed region) - what a learner that keeps the policy on the GPU pays."""
    import torch
    import torch.distributed as dist
    from amp_extensions_b200 import VecSimEnv
    from amp_extensions_b200.rollout import DeviceRollout
    pool = ds.states[:4096] * 0.3
    pool[:, 0] = 1.5
    env = VecSimEnv(ens, E, horizon=300, reset_states=pool, seed=1, cost=cost)
    env.reset()
    ro = DeviceRollout(env, _Policy(S_DIM, A_DIM), seed=0)
    from amp_extensions_b200.rollout import HostPathStream, RolloutBatch
    dl = HostPathStream(device)
    # two device batches alternate (collect k+1 fills one while the other one's paths cross PCIe): no allocation in the loop
    use_cost = env.cost is not None and getattr(env, "_w_dev", None) is not None
    batches = [RolloutBatch(ro.eng, horizon, E, S_DIM, A_DIM, use_cost) for _ in range(2)]
    ro.collect(horizon, batch=batches[0])
    for k in range(4):                          # both pinned slots exist before the clock starts
        dl.submit(ro.collect(horizon, batch=batches[k % 2]))
        if k > 0:
            dl.collect()
    dl.collect()
    torch.cuda.synchronize(device)
    barrier()
    t0 = time.perf_counter()
    for i in range(iters):
        dl.submit(ro.collect(horizon, batch=batches[i % 2]))   # horizon i computes while horizon i-1 crosses PCIe
        if i > 0:
            _ = float(dl.collect()["rewards"][0, 0])
    _ = float(dl.collect()["rewards"][0, 0])
    torch.cuda.synchronize(device)
    dt = torch.tensor([time.perf_counter() - t0], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    return {"value": E * world * horizon * iters / float(dt.item()), "unit": UNIT, "horizon": horizon, "horizons": iters,
            "d2h_bytes_per_horizon": dl.bytes_per_batch, "h2d_bytes_per_step": 0,
            "api": "amp_extensions_b200.rollout.DeviceRollout.collect + rollout.HostPathStream: the paths of a horizon "
                   "are downloaded to pinned host memory (one piece per horizon, inside the timed region) while the next "
                   "horizon computes; the last download is exposed"}


def plugin_single_env(ens, ds, device, n=200):
    """The UNCHANGED sampler's calling pattern (milo/milo/sampler.py:48-66): one env, one SimEnv.step per call, numpy
    float64 observation in and out - through the plugin on the GPU."""
    import numpy as np
    from amp_extensions_b200 import SimEnv
    env = SimEnv(ens, reset_states=(ds.states[:64] * 0.3 + 0.5).numpy(), seed=0)
    env.reset()
    rng = np.random.default_rng(0)
    acts = rng.standard_normal((n + 20, A_DIM))
    for i in range(20):
        env.step(acts[i])
    t0 = time.perf_counter()
    for i in range(n):
        ob, r, d, info = env.step(acts[20 + i])
        if d:
            env.reset()
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": UNIT, "us_per_step": dt / n * 1e6,
            "api": "amp_extensions_b200.SimEnv.step (numpy float64 [226] in / out, one env per call)",
            "graph": bool(getattr(env, "_fast", None) is not None and env._fast.graph is not None)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default: 500; 30 with --config 4 / 5)")
    ap.add_argument("--warmup", type=int, default=None, help="untimed steps first, at least 3 (default: 20; 5 with "
                                                              "--config 4 / 5)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS),
                    help="BASELINE.json workload, 1-based: 2 = configs[1] (default, the headline), 3 = imitation only, "
                         "4 = 1 M envs + imitation + quantile, 5 = 8 x (1024 x 4) at 512 Ki envs per GPU")
    ap.add_argument("--precision", default="fp16", choices=["fp16", "tf32", "bf16"])
    ap.add_argument("--envs", type=int, default=None, help="envs per GPU per step (default: the config's)")
    ap.add_argument("--e2e-chunks", type=int, default=2)
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true", help="profiling runs only: no host-buffer pass")
    ap.add_argument("--skip-sustained", action="store_true")
    ap.add_argument("--skip-extras", action="store_true", help="no device-policy rollout / single-env plugin timing")
    ap.add_argument("--rff-split", default="auto", choices=["auto", "on", "off"],
                    help="hi/lo operand pairs in the cost-feature GEMM: measured decision (auto), always, never")
    ap.add_argument("--graph-check", action="store_true", help="also time the steps replayed from CUDA graphs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs as DIR/<name>.npy (at most 64 MB in all)")
    args = ap.parse_args()
    long_steps = args.config in (4, 5)  # a step is 20-60 ms here
    if args.steps is None:
        args.steps = 30 if long_steps else 500
    if args.warmup is None:
        args.warmup = 5 if long_steps else 20
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the CUDA path's outputs (--impl ours)")
    # The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner on
    # stdout when NCCL_DEBUG is set on the box), so file descriptor 1 is pointed at stderr for the duration of the
    # run and the JSON line goes to the original stdout.
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


_JSON_OUT = None


def emit(line):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


if __name__ == "__main__":
    sys.exit(main())
