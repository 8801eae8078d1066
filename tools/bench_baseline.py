"""Benchmark of the MLP value baseline (DESIGN.md section 9, row f6): predict and one epoch of fit_data at the MILO
shape, against the same loop in float32 torch on the same GPU (eager, and replayed from CUDA graphs) and on the host's
cores.

Workload: 40 000 envs x 32 steps = 1 280 000 rows, S = 226, hidden (128, 128), batch 64, one epoch = 19 999 Adam steps.
The torch arms read a materialised float32 feature matrix (1.2 GB; the device path forms features on the fly), so they
measure the optimiser loop alone.  Every GPU time is taken between CUDA events after a synchronise.

  python tools/bench_baseline.py --out profiles/r03_baseline_bench.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


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


def features(obs, t):
    o = torch.clamp(obs.double(), -10, 10) / 10.0
    a = (t.double() / 1000.0).unsqueeze(1)
    return torch.cat([o, a, a ** 2, a ** 3, a ** 4], dim=1).float()


def torch_step_fn(model, opt, x, y, bs):
    loss_fn = torch.nn.MSELoss()

    def step(idx):
        opt.zero_grad()
        loss = loss_fn(model(x[idx]), y[idx])
        loss.backward()
        opt.step()
    return step


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=40_000)
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--obs", type=int, default=226)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--cpu-steps", type=int, default=300, help="steps of the host loop that are timed")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from amp_extensions_b200.baseline import DeviceMLPBaseline, MLPBaseline
    from amp_extensions_b200.engine import Engine

    assert torch.cuda.is_available(), "bench_baseline measures on the GPU"
    S, bs = args.obs, args.batch
    n = args.envs * args.steps
    nb = max(0, n // bs - 1)
    g = torch.Generator(device="cuda").manual_seed(0)
    obs = (4.0 * torch.randn(n, S, device="cuda", generator=g)).contiguous()
    t = (torch.arange(n, device="cuda", dtype=torch.int32) // args.envs).contiguous()   # time-major rows
    y = (torch.tanh(obs[:, :5]).sum(1) + 0.3 * torch.randn(n, device="cuda", generator=g)).contiguous()
    perm = torch.randperm(n, device="cuda", generator=g)

    class Spec:
        observation_dim = S

    torch.manual_seed(0)
    host = MLPBaseline(Spec(), batch_size=bs)
    init = [p.detach().clone() for p in host.model.parameters()]
    eng = Engine(state_dim=8, action_dim=0, num_models=1, hidden_sizes=[], transform=False)
    vf = DeviceMLPBaseline(eng, host)
    s0 = eng.baseline_read()
    res = {"workload": dict(rows=n, envs=args.envs, steps=args.steps, obs_dim=S, hidden=[128, 128], batch=bs,
                            adam_steps=nb), "card": card()}

    # predict: all rows, then the warm-up is repeated five times
    out = torch.empty(n, device="cuda")
    eng.baseline_predict(obs, t, out)
    res["predict_s"] = gpu_timed(lambda: eng.baseline_predict(obs, t, out), reps=5)

    def restore():
        eng.baseline_state(params=s0["params"], exp_avg=s0["exp_avg"], exp_avg_sq=s0["exp_avg_sq"], step=s0["step"])

    # device fit, eager enqueue of the whole epoch (one warm-up epoch first)
    eng.baseline_fit(obs, t, y, perm, nb)
    restore()
    res["device_fit_eager_s"] = gpu_timed(lambda: eng.baseline_fit(obs, t, y, perm, nb))
    p_eager = eng.baseline_read()["params"]
    # device fit replayed from graphs of K steps (a restarting chunk, then continuing ones)
    K = 500
    restore()
    torch.cuda.synchronize()
    g_first, g_next = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
    with torch.cuda.graph(g_first):
        eng.baseline_fit(obs, t, y, perm, K, restart=True)
    with torch.cuda.graph(g_next):
        eng.baseline_fit(obs, t, y, perm, K, restart=False)
    chunks = -(-nb // K)

    def replay():
        g_first.replay()
        for _ in range(chunks - 1):
            g_next.replay()
    restore()
    replay()                       # warm-up replay
    restore()
    res["device_fit_graph_s"] = gpu_timed(replay)
    p_graph = eng.baseline_read()["params"]
    res["device_graph_equals_eager"] = bool(torch.equal(p_eager, p_graph))
    res["device_us_per_step_eager"] = 1e6 * res["device_fit_eager_s"] / nb
    res["device_us_per_step_graph"] = 1e6 * res["device_fit_graph_s"] / nb

    # the same loop in float32 torch on the GPU
    x = features(obs, t)
    yy = y.reshape(-1, 1)

    def fresh(device, capturable=False):
        m = MLPBaseline(Spec(), batch_size=bs).model.to(device)
        with torch.no_grad():
            for p, q in zip(m.parameters(), init):
                p.copy_(q)
        return m, torch.optim.Adam(m.parameters(), lr=1e-3, capturable=capturable)

    model, opt = fresh("cuda")
    step = torch_step_fn(model, opt, x, yy, bs)
    for mb in range(20):
        step(perm[mb * bs:(mb + 1) * bs])

    def torch_epoch():
        for mb in range(nb):
            step(perm[mb * bs:(mb + 1) * bs])
    model, opt = fresh("cuda")
    step = torch_step_fn(model, opt, x, yy, bs)
    res["torch_gpu_eager_s"] = gpu_timed(torch_epoch)
    res["torch_gpu_eager_us_per_step"] = 1e6 * res["torch_gpu_eager_s"] / nb
    p_torch = torch.cat([p.detach().reshape(-1) for p in model.parameters()])
    res["device_vs_torch_params_max_abs"] = float((p_torch - p_eager).abs().max())
    try:
        model, opt = fresh("cuda", capturable=True)
        step = torch_step_fn(model, opt, x, yy, bs)
        KT = 100
        pstat = torch.empty(KT * bs, device="cuda", dtype=torch.int64)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            pstat.copy_(perm[:KT * bs])
            for j in range(3):
                step(pstat[j * bs:(j + 1) * bs])
        torch.cuda.current_stream().wait_stream(side)
        gt = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gt):
            for j in range(KT):
                step(pstat[j * bs:(j + 1) * bs])
        full = nb // KT

        def torch_graph_epoch():
            for c in range(full):
                pstat.copy_(perm[c * KT * bs:(c + 1) * KT * bs])
                gt.replay()
        torch_graph_epoch()
        res["torch_gpu_graph_s"] = gpu_timed(torch_graph_epoch) * nb / (full * KT)
        res["torch_gpu_graph_us_per_step"] = 1e6 * res["torch_gpu_graph_s"] / nb
        res["torch_gpu_graph_note"] = f"graphs of {KT} steps; {full * KT} of {nb} steps timed, scaled to the epoch"
    except Exception as e:  # noqa: BLE001 - reported, not hidden
        res["torch_gpu_graph_error"] = repr(e)

    # the same loop on the host's cores
    xc, yc, pc = x[:200_000].cpu(), yy[:200_000].cpu(), torch.randperm(200_000)
    model, opt = fresh("cpu")
    step = torch_step_fn(model, opt, xc, yc, bs)
    for mb in range(20):
        step(pc[mb * bs:(mb + 1) * bs])
    t0 = time.perf_counter()
    for mb in range(args.cpu_steps):
        step(pc[mb * bs:(mb + 1) * bs])
    per = (time.perf_counter() - t0) / args.cpu_steps
    res["torch_cpu_us_per_step"] = 1e6 * per
    res["torch_cpu_epoch_s_extrapolated"] = per * nb
    res["torch_cpu_threads"] = torch.get_num_threads()
    res["torch_cpu_note"] = f"{args.cpu_steps} steps timed, extrapolated to {nb}"

    best_dev = min(res["device_fit_eager_s"], res["device_fit_graph_s"])
    res["speedup_vs_torch_gpu_eager"] = res["torch_gpu_eager_s"] / best_dev
    if "torch_gpu_graph_s" in res:
        res["speedup_vs_torch_gpu_graph"] = res["torch_gpu_graph_s"] / best_dev
    res["speedup_vs_torch_cpu"] = res["torch_cpu_epoch_s_extrapolated"] / best_dev
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
