"""Latency of parallel.global_quantile on one GPU (VERDICT r1 item 9: < 1 ms per call at 1 M samples).

    python tools/bench_quantile.py [--n 1048576] [--reps 50]

Prints one JSON line: the GPU's name and power limit, then per input (uniform, 90 % exact zeros, lognormal with
sigma 6) the ms per call (host wall around the call, device idle before it), the library launches per call, and
whether the results at q = 0.1, 0.5, 0.9 equal the float64 sort reference (torch.quantile where n <= 2^24).
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


def inputs(n, g):
    """The timed inputs: smooth control, heavy ties (every sample of a warp in one bin), 25 decades of spread."""
    return {
        "uniform": torch.rand(n, device="cuda", generator=g) ** 2,
        "zeros90": torch.where(torch.rand(n, device="cuda", generator=g) < 0.9, 0.0,
                               torch.rand(n, device="cuda", generator=g)),
        "lognormal6": torch.exp(6.0 * torch.randn(n, device="cuda", generator=g, dtype=torch.float64)).float(),
    }


def reference(x, q):
    xs = torch.sort(x.double().cpu()).values
    pos = q * (xs.numel() - 1)
    k0 = math.floor(pos)
    v0, v1 = xs[k0], xs[min(k0 + 1, xs.numel() - 1)]
    return float(v0) if pos == k0 else float(torch.lerp(v0, v1, pos - k0))


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        return torch.cuda.get_device_name()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 20)
    ap.add_argument("--reps", type=int, default=50)
    args = ap.parse_args()
    from amp_extensions_b200 import _lib, parallel
    from amp_extensions_b200.engine import Engine
    eng = Engine(8, 2, 2, [16], precision="fp16")
    g = torch.Generator(device="cuda").manual_seed(0)
    res = {"gpu": gpu_info(), "n": args.n, "reps": args.reps}
    for name, x in inputs(args.n, g).items():
        check = {}
        for q in (0.1, 0.5, 0.9):
            got, ref = parallel.global_quantile(x, q, engine=eng), reference(x, q)
            check[f"q{q}"] = {"got": got, "ref": ref, "ulps": abs(got - ref) / math.ulp(ref) if ref else abs(got)}
        torch.cuda.synchronize()
        l0 = _lib.launch_count()
        t0 = time.perf_counter()
        for _ in range(args.reps):
            parallel.global_quantile(x, 0.9, engine=eng)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / args.reps
        res[name] = {"ms_per_call": dt * 1e3, "library_launches_per_call": (_lib.launch_count() - l0) / args.reps,
                     "check": check}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
