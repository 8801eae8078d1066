"""Timing of the on-device NPG step (DeviceNPG.update) and of its Fisher-vector product for the MILO policy
(226 -> 32 -> 32 -> 28 tanh), against the same math in torch autograd on the same GPU and on the host CPU.

    python tools/bench_npg.py [--out profiles/npg_bench.json]

Prints one JSON line.  Times are medians of CUDA-event timings after warm-up (host arm: median of five wall-clock
products after one warm-up, torch threads, at most 131 072 rows).  The FP32-pipe fraction counts the Fisher-vector product's multiply-adds from the layer shapes (JVP through every layer
including the bias column, backward data products of the hidden layers, weight / bias gradients) at 2 FLOP each, over
148 SMs x 128 FP32 lanes x the card's maximum SM clock read in the same run.
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

SIZES = [226, 32, 32, 28]


def fvp_macs(sizes):
    L = len(sizes) - 1
    jvp = sum((sizes[l] + 1) * sizes[l + 1] + (sizes[l] * sizes[l + 1] if l > 0 else 0) for l in range(L))
    bwd = sum(sizes[l] * sizes[l + 1] for l in range(1, L))
    wgrad = sum((sizes[l] + 1) * sizes[l + 1] for l in range(L))
    return jvp + bwd + wgrad


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, power, clock = [x.strip() for x in q.split(",")]
    return name, float(power), float(clock)


def events(fn, reps):
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return ts[len(ts) // 2]


def torch_arm(sizes, obs, act, adv, dev, cg_iters=10, damping=1e-4, delta=0.01):
    """mjrl's NPG step in torch autograd (fp32): flat_vpg, cg_solve over HVP (double backward of mean_kl), step."""
    g = torch.Generator(device="cpu").manual_seed(0)
    params = []
    for i, o in zip(sizes[:-1], sizes[1:]):
        params += [(torch.randn(o, i, generator=g) / i ** 0.5).to(dev), torch.zeros(o).to(dev)]
    params.append(torch.full((sizes[-1],), -0.5).to(dev))
    theta = torch.cat([p.reshape(-1) for p in params])

    def unflat(t):
        out, off = [], 0
        for p in params:
            out.append(t[off:off + p.numel()].reshape(p.shape)); off += p.numel()
        return out

    def mean(t):
        ps = unflat(t)
        h = obs
        for k in range(0, len(ps) - 3, 2):
            h = torch.tanh(h @ ps[k].T + ps[k + 1])
        return h @ ps[-3].T + ps[-2], ps[-1]

    def hvp(v, t0):
        t = t0.clone().requires_grad_(True)
        mn, ln = mean(t)
        with torch.no_grad():
            mo, lo = mean(t0)
        kl = (((mo - mn) ** 2 + torch.exp(lo) ** 2 - torch.exp(ln) ** 2) / (2 * torch.exp(ln) ** 2 + 1e-8) + ln - lo).sum(1).mean()
        gk = torch.autograd.grad(kl, t, create_graph=True)[0]
        return torch.autograd.grad((gk * v).sum(), t)[0] + damping * v

    def update():
        t = theta.clone().requires_grad_(True)
        mu, ls = mean(t)
        ll = -0.5 * (((act - mu) / torch.exp(ls)) ** 2).sum(1) - ls.sum()
        s = (torch.exp(ll - ll.detach()) * adv).mean()
        gr = torch.autograd.grad(s, t)[0]
        x = torch.zeros_like(gr); r = gr.clone(); p = gr.clone(); rr = r.dot(r)
        for _ in range(cg_iters):
            z = hvp(p, theta)
            v = rr / p.dot(z)
            x += v * p; r -= v * z
            nr = r.dot(r); p = r + nr / rr * p; rr = nr
        alpha = torch.sqrt(torch.abs(delta / (gr.dot(x) + 1e-10)))
        return theta + alpha * x

    v = torch.randn(theta.numel(), device=dev)
    return (lambda: hvp(v, theta)), update


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=11)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_npg.py measures on the GPU"
    from amp_extensions_b200 import Engine
    from amp_extensions_b200.npg import DeviceNPG
    name, power, clock_mhz = gpu_info()
    macs = fvp_macs(SIZES)
    peak = 148 * 128 * 2 * clock_mhz * 1e6
    res = dict(card=name, power_limit_w=power, sm_clock_max_mhz=clock_mhz, policy=SIZES, fvp_macs_per_row=macs, sizes=[])
    for envs in (1024, 40_000):
        n = envs * 32
        g = torch.Generator(device="cuda").manual_seed(0)
        obs = torch.randn(n, SIZES[0], device="cuda", generator=g)
        act = 0.3 * torch.randn(n, SIZES[-1], device="cuda", generator=g)
        adv = torch.randn(n, device="cuda", generator=g)
        eng = Engine(SIZES[0], SIZES[-1], 1, [32])   # a handle to hold the policy; no ensemble is loaded
        sys.path.insert(0, os.path.join(ROOT, "examples"))
        from milo_iteration import GaussianMLP
        pol = GaussianMLP(SIZES[0], SIZES[-1], hidden=tuple(SIZES[1:-1]))
        npg = DeviceNPG(eng, pol)
        theta0 = npg.params().clone()

        def upd():
            eng.npg_params(theta0)
            npg.update((obs, act), adv)
        for _ in range(3):
            upd()
        t_update = events(upd, args.reps)
        eng.npg_prepare(obs)
        v = torch.randn(npg.n_params, device="cuda", dtype=torch.float64)
        out = torch.empty(npg.n_params + 2, device="cuda", dtype=torch.float64)
        for _ in range(3):
            eng.npg_fvp(obs, v=v, out=out)
        t_fvp = events(lambda: eng.npg_fvp(obs, v=v, out=out), args.reps * 3)
        t_fvp_bound = 2.0 * macs * n / peak * 1e3
        hv, tupd = torch_arm(SIZES, obs, act, adv, "cuda")
        for _ in range(2):
            hv(); tupd()
        t_torch_fvp = events(hv, args.reps)
        t_torch_update = events(tupd, max(3, args.reps // 2))
        cpu_n = min(n, 131_072)
        hc, uc = torch_arm(SIZES, obs[:cpu_n].cpu(), act[:cpu_n].cpu(), adv[:cpu_n].cpu(), "cpu")
        hc()
        cpu_ts = []
        for _ in range(5):
            t0 = time.perf_counter()
            hc()
            cpu_ts.append((time.perf_counter() - t0) * 1e3)
        t_cpu_fvp = sorted(cpu_ts)[len(cpu_ts) // 2]
        res["sizes"].append(dict(
            rows=n, update_ms=round(t_update, 3), fvp_ms=round(t_fvp, 4), fvp_fp32_bound_ms=round(t_fvp_bound, 4),
            fvp_fp32_pipe_fraction=round(t_fvp_bound / t_fvp, 3), fvp_gflops=round(2.0 * macs * n / t_fvp / 1e6, 1),
            torch_gpu_fvp_ms=round(t_torch_fvp, 3), torch_gpu_update_ms=round(t_torch_update, 3),
            update_speedup_vs_torch_gpu=round(t_torch_update / t_update, 2),
            cpu_torch_fvp_ms=round(t_cpu_fvp, 1), cpu_rows=cpu_n, cpu_threads=torch.get_num_threads()))
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
