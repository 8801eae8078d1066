"""Benchmark of behaviour cloning (DESIGN.md section 9, row f7): one epoch of BC.fit on the MILO policy (226 -> 32 -> 32
-> 28 tanh), batch 64, both losses, at 100 000 and 1 000 000 expert rows, against the same loop in float32 torch on the
same GPU (eager, and replayed from CUDA graphs) and on the host's cores.

An epoch is int(n / 64) Adam steps (1 562 and 15 625) on minibatches drawn with replacement.  Every GPU time is taken
between CUDA events after a synchronise; the card's name and power limit are read in the same run.

  python tools/bench_bc.py --out profiles/r03_bc_bench.json
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SIZES = (226, 32, 32, 28)


def gpu_timed(fn, reps=1):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps / 1e3


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True)
    return {"name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip()}


class Policy:
    """mjrl's MLP attributes with identity transformations."""

    def __init__(self, seed=0):
        g = torch.Generator().manual_seed(seed)

        class Net:
            pass
        self.model = Net()
        self.model.fc_layers = [torch.nn.Linear(SIZES[i], SIZES[i + 1]) for i in range(len(SIZES) - 1)]
        for l in self.model.fc_layers:
            l.weight.data = torch.randn(l.weight.shape, generator=g) / math.sqrt(l.weight.shape[1])
            l.bias.data.zero_()
        self.model.nonlinearity = torch.tanh
        self.model.in_shift, self.model.in_scale = torch.zeros(SIZES[0]), torch.ones(SIZES[0])
        self.model.out_shift, self.model.out_scale = torch.zeros(SIZES[-1]), torch.ones(SIZES[-1])
        self.log_std = torch.full((SIZES[-1],), -0.5)


def torch_step_fn(policy, device, loss_type, obs, act, capturable=False):
    layers = [torch.nn.Linear(l.in_features, l.out_features).to(device) for l in policy.model.fc_layers]
    with torch.no_grad():
        for dst, src in zip(layers, policy.model.fc_layers):
            dst.weight.copy_(src.weight)
            dst.bias.copy_(src.bias)
    log_std = torch.nn.Parameter(policy.log_std.clone().to(device))
    params = [p for l in layers for p in l.parameters()] + [log_std]
    opt = torch.optim.Adam(params, lr=1e-3, capturable=capturable)
    mse = torch.nn.MSELoss()

    def step(idx):
        o, a = obs[idx], act[idx]
        x = o
        for l in layers[:-1]:
            x = torch.tanh(l(x))
        mu = layers[-1](x)
        if loss_type == "MSE":
            lo = mse(mu, a)
        else:
            z = (a - mu) / torch.exp(log_std)
            lo = -torch.mean(-0.5 * torch.sum(z ** 2, dim=1) - torch.sum(log_std) - 0.5 * SIZES[-1] * math.log(2 * math.pi))
        opt.zero_grad()
        lo.backward()
        opt.step()
    return step


def bench_case(n, loss_type, cpu_steps):
    from amp_extensions_b200.bc import DeviceBC
    from amp_extensions_b200.engine import Engine
    bs = 64
    steps = n // bs
    g = torch.Generator(device="cuda").manual_seed(n)
    obs = torch.randn(n, SIZES[0], device="cuda", generator=g).contiguous()
    act = (0.5 * torch.randn(n, SIZES[-1], device="cuda", generator=g)).contiguous()
    idx = torch.randint(0, n, (steps * bs,), device="cuda", generator=g)
    eng = Engine(state_dim=8, action_dim=0, num_models=1, hidden_sizes=[], transform=False)
    policy = Policy()
    bc = DeviceBC(eng, policy, epochs=1, batch_size=bs, loss_type=loss_type)
    s0 = eng.bc_read()
    res = {"rows": n, "loss": loss_type, "batch": bs, "adam_steps": steps}

    def restore():
        eng.bc_state(params=s0["params"], exp_avg=s0["exp_avg"], exp_avg_sq=s0["exp_avg_sq"], step=s0["step"])

    eng.bc_fit(obs, act, idx, steps)                       # warm-up epoch
    restore()
    res["device_fit_eager_s"] = gpu_timed(lambda: eng.bc_fit(obs, act, idx, steps))
    p_eager = eng.bc_read()["params"]
    K = 500
    restore()
    torch.cuda.synchronize()
    g_first, g_next = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
    with torch.cuda.graph(g_first):
        eng.bc_fit(obs, act, idx, K, restart=True)
    with torch.cuda.graph(g_next):
        eng.bc_fit(obs, act, idx, K, restart=False)
    chunks = -(-steps // K)

    def replay():
        g_first.replay()
        for _ in range(chunks - 1):
            g_next.replay()
    restore()
    replay()
    restore()
    res["device_fit_graph_s"] = gpu_timed(replay)
    res["device_graph_equals_eager"] = bool(torch.equal(p_eager, eng.bc_read()["params"]))
    res["device_us_per_step_eager"] = 1e6 * res["device_fit_eager_s"] / steps
    res["device_us_per_step_graph"] = 1e6 * res["device_fit_graph_s"] / steps
    res["device_loss_s"] = gpu_timed(lambda: bc.loss(obs, act), reps=5)

    step = torch_step_fn(policy, "cuda", loss_type, obs, act)
    for j in range(20):
        step(idx[j * bs:(j + 1) * bs])
    step = torch_step_fn(policy, "cuda", loss_type, obs, act)

    def torch_epoch():
        for j in range(steps):
            step(idx[j * bs:(j + 1) * bs])
    res["torch_gpu_eager_s"] = gpu_timed(torch_epoch)
    res["torch_gpu_eager_us_per_step"] = 1e6 * res["torch_gpu_eager_s"] / steps
    try:
        step = torch_step_fn(policy, "cuda", loss_type, obs, act, capturable=True)
        KT = 100
        pstat = torch.empty(KT * bs, device="cuda", dtype=torch.int64)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            pstat.copy_(idx[:KT * bs])
            for j in range(3):
                step(pstat[j * bs:(j + 1) * bs])
        torch.cuda.current_stream().wait_stream(side)
        gt = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gt):
            for j in range(KT):
                step(pstat[j * bs:(j + 1) * bs])
        full = steps // KT

        def torch_graph_epoch():
            for c in range(full):
                pstat.copy_(idx[c * KT * bs:(c + 1) * KT * bs])
                gt.replay()
        torch_graph_epoch()
        res["torch_gpu_graph_s"] = gpu_timed(torch_graph_epoch) * steps / (full * KT)
        res["torch_gpu_graph_us_per_step"] = 1e6 * res["torch_gpu_graph_s"] / steps
        res["torch_gpu_graph_note"] = f"graphs of {KT} steps; {full * KT} of {steps} steps timed, scaled to the epoch"
    except Exception as e:  # noqa: BLE001 - reported, not hidden
        res["torch_gpu_graph_error"] = repr(e)

    oc, ac, ic = obs[:100_000].cpu(), act[:100_000].cpu(), torch.randint(0, min(n, 100_000), (cpu_steps + 20, bs))
    step = torch_step_fn(policy, "cpu", loss_type, oc, ac)
    for j in range(20):
        step(ic[j])
    t0 = time.perf_counter()
    for j in range(cpu_steps):
        step(ic[20 + j])
    per = (time.perf_counter() - t0) / cpu_steps
    res["torch_cpu_us_per_step"] = 1e6 * per
    res["torch_cpu_epoch_s_extrapolated"] = per * steps
    res["torch_cpu_threads"] = torch.get_num_threads()
    res["torch_cpu_note"] = f"{cpu_steps} steps timed, extrapolated to {steps}"
    best = min(res["device_fit_eager_s"], res["device_fit_graph_s"])
    res["speedup_eager_vs_torch_gpu_eager"] = res["torch_gpu_eager_s"] / res["device_fit_eager_s"]
    if "torch_gpu_graph_s" in res:
        res["speedup_graph_vs_torch_gpu_graph"] = res["torch_gpu_graph_s"] / res["device_fit_graph_s"]
    res["speedup_vs_torch_cpu"] = res["torch_cpu_epoch_s_extrapolated"] / best
    eng.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, nargs="+", default=[100_000, 1_000_000])
    ap.add_argument("--cpu-steps", type=int, default=300, help="steps of the host loop that are timed")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_bc measures on the GPU"
    res = {"workload": dict(policy=list(SIZES), nonlinearity="tanh", batch=64, epochs=1), "card": card(), "cases": []}
    for n in args.rows:
        for loss in ("MSE", "MLE"):
            res["cases"].append(bench_case(n, loss, args.cpu_steps))
            print(json.dumps(res["cases"][-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
