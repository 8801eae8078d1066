"""parallel.global_quantile against float64 order statistics, on data where a histogram quantile goes wrong: heavy
ties, a few huge outliers, lognormal spread over 25 decades, infinities, NaN, signed zeros, subnormals next to
FLT_MAX, values on bin edges.  Also simstep_reduce_max_sum (the dataset-maximum threshold) against numpy float64.

The contract (global_quantile's docstring):
  * any NaN in the union of the samples, or no samples at all, gives NaN;
  * q outside [0, 1] raises ValueError;
  * with pos = q * (n - 1), k0 = floor(pos), w = pos - k0: w == 0 gives sorted[k0] exactly (also where
    torch.quantile returns NaN from lerp(inf, inf, 0)), w != 0 gives torch.quantile's lerp within 2 float64 ulp,
    NaN exactly where it is NaN, the same infinity where it is infinite (torch's lerp is FMA-fused on some builds,
    so its last bit is build-dependent);
  * repeated calls are bit-identical, and every rank gets the same value.

CPU tests (torch path, one process and two gloo ranks with uneven and empty shards) run anywhere; the device path
(simstep_quantile_op) and the max/sum kernel need a GPU."""
import math
import os
import socket
import struct
import sys
import tempfile

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from amp_extensions_b200 import parallel

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FLT_MAX = float(np.finfo(np.float32).max)
CASES = ("uniform", "lognormal6", "outlier", "posinf", "bothinf", "allinf", "nan", "ties", "zeros90", "constant",
         "mixedsign", "subnormal_max", "binedges")
SIZES = (0, 1, 2, 3, 4097, 1_000_003)
QS = (0.0, 0.1, 0.5, 0.9, 0.999, 1.0)
TORCH_QUANTILE_MAX = 1 << 24  # torch.quantile refuses larger inputs


def make_case(name, n, seed=0):
    """fp32 CPU samples of one adversarial distribution (deterministic in name, n, seed)."""
    g = torch.Generator().manual_seed(1000 * seed + CASES.index(name))
    u = torch.rand(n, generator=g)
    pick = lambda: int(torch.randint(0, n, (1,), generator=g))  # noqa: E731
    if name == "uniform":
        x = u
    elif name == "lognormal6":
        x = torch.exp(6.0 * torch.randn(n, generator=g, dtype=torch.float64)).float()
    elif name == "outlier":
        x = torch.randn(n, generator=g).abs() * 0.05
        if n:
            x[pick()] = 1e6
    elif name == "posinf":
        x = u
        if n:
            x[pick()] = math.inf
    elif name == "bothinf":
        x = u
        if n:
            i = pick()
            x[i] = -math.inf
            if n > 1:
                x[(i + 1 + pick() % (n - 1)) % n] = math.inf
    elif name == "allinf":
        x = torch.full((n,), math.inf)
    elif name == "nan":
        x = u
        if n:
            x[pick()] = math.nan
    elif name == "ties":
        x = torch.randint(0, 10, (n,), generator=g).float()
    elif name == "zeros90":
        x = torch.where(u < 0.9, torch.zeros(()), torch.rand(n, generator=g))
    elif name == "constant":
        x = torch.full((n,), 3.25)
    elif name == "mixedsign":
        x = torch.randn(n, generator=g)
        x = torch.where(u < 0.1, torch.tensor(-0.0), torch.where(u > 0.9, torch.tensor(0.0), x))
    elif name == "subnormal_max":
        vals = torch.tensor([1e-40, 2e-40, -3e-42, 1.4e-45, 1.0, 3e38, FLT_MAX, -FLT_MAX], dtype=torch.float32)
        x = vals[torch.randint(0, vals.numel(), (n,), generator=g)]
    elif name == "binedges":
        x = torch.randint(0, 4097, (n,), generator=g).float() / 4096.0
    else:
        raise ValueError(name)
    assert x.dtype == torch.float32 and x.numel() == n
    return x.contiguous()


def exact_qs(n):
    """q values with w == 0 beyond 0 and 1: j / 2^m when n = 2^m + 1."""
    m = n - 1
    if m < 2 or m & (m - 1):
        return ()
    return tuple(j / m for j in sorted({1, m // 3, m // 2, m - 1}))


def ref_order_stats(xs_sorted, q):
    """(sorted[k0], sorted[k1], w) of the float64 samples sorted over all ranks: pos = q (n - 1)."""
    n = xs_sorted.size
    pos = q * (n - 1)
    k0 = math.floor(pos)
    k1 = min(k0 + 1, n - 1)
    return float(xs_sorted[k0]), float(xs_sorted[k1]), pos - k0


def bits(v):
    return struct.pack("<d", v)


def check_quantile(got, x, q, tq=None, xs_sorted=None):
    """Assert the contract of the module docstring for one result `got` of the samples x (any float dtype, any
    device, the union over all ranks) at q; tq: torch.quantile of x.double() at q when already computed."""
    xd = x.detach().double().cpu().reshape(-1)
    n = xd.numel()
    if n == 0 or bool(torch.isnan(xd).any()):
        assert math.isnan(got), (q, got)
        return
    if xs_sorted is None:
        xs_sorted = np.sort(xd.numpy())
    v0, v1, w = ref_order_stats(xs_sorted, q)
    if tq is None and n <= TORCH_QUANTILE_MAX:
        tq = float(torch.quantile(xd, q))
    if w == 0.0:
        assert got == v0, (q, got, v0)
        if tq is not None:  # the documented deviation: lerp(inf, inf, 0) is NaN in torch, sorted[k0] here
            assert got == tq or (math.isnan(tq) and math.isinf(v0)), (q, got, tq)
        return
    ref = tq if tq is not None else float(torch.lerp(torch.tensor(v0, dtype=torch.float64),
                                                     torch.tensor(v1, dtype=torch.float64), w))
    if math.isnan(ref):
        assert math.isnan(got), (q, got, v0, v1, w)
    elif math.isinf(ref):
        assert got == ref, (q, got, ref)
    else:
        assert abs(got - ref) <= 2 * math.ulp(ref), (q, got, ref, (got - ref) / math.ulp(ref))


def check_all_qs(x, quantile_fn, qs=None):
    """quantile_fn(q) over QS and the exact q values of x's size, each checked against the float64 references."""
    xd = x.detach().double().cpu().reshape(-1)
    qs = tuple(QS if qs is None else qs) + exact_qs(xd.numel())
    xs_sorted = np.sort(xd.numpy())
    tqs = [None] * len(qs)
    if 0 < xd.numel() <= TORCH_QUANTILE_MAX:
        tqs = torch.quantile(xd, torch.tensor(qs, dtype=torch.float64)).tolist()
    for q, tq in zip(qs, tqs):
        check_quantile(quantile_fn(q), x, q, tq=tq, xs_sorted=xs_sorted)


# ---- torch path, one process ------------------------------------------------------------------------------------

@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("case", CASES)
def test_torch_path_fp32_matches_float64_order_statistics(case, n):
    x = make_case(case, n)
    check_all_qs(x, lambda q: parallel.global_quantile(x, q))


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("case", CASES + ("fine64",))
def test_torch_path_fp64_matches_float64_order_statistics(case, n):
    """fp64 samples take the 64-bit key; fine64 differs only below fp32 resolution, so a key that dropped the low
    32 bits (or rounded to fp32) would pick the wrong sample."""
    if case == "fine64":
        g = torch.Generator().manual_seed(5)
        x = 1.0 + torch.randint(0, 1 << 20, (n,), generator=g).double() * 2.0 ** -52
    else:
        x = make_case(case, n).double()
    check_all_qs(x, lambda q: parallel.global_quantile(x, q))


def test_other_dtypes_go_through_fp64():
    x = make_case("ties", 4097).to(torch.int32)
    check_all_qs(x, lambda q: parallel.global_quantile(x, q))
    h = make_case("uniform", 4097).half()
    check_all_qs(h, lambda q: parallel.global_quantile(h, q))


@pytest.mark.parametrize("q", [-0.1, 1.0000001, math.nan, math.inf])
def test_q_outside_unit_interval_raises(q):
    with pytest.raises(ValueError):
        parallel.global_quantile(make_case("uniform", 10), q)


def test_repeated_calls_are_bit_identical():
    for case in ("lognormal6", "zeros90", "mixedsign", "subnormal_max"):
        x = make_case(case, 4097)
        for q in (0.1, 0.5, 0.9):
            assert bits(parallel.global_quantile(x, q)) == bits(parallel.global_quantile(x, q)), (case, q)


# ---- torch path, two gloo ranks -------------------------------------------------------------------------------

GLOO_SIZES = (0, 1, 3, 4097)
GLOO_LARGE = ("lognormal6", "zeros90", "nan")


def _splits(n):
    """Shard boundaries of rank 0 / rank 1: uneven, rank 0 empty, rank 1 empty."""
    return (n // 3, 0, n)


def _gloo_worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(2)  # two ranks share the host
    from amp_extensions_b200 import parallel as par
    res = {}
    jobs = [(c, n) for c in CASES for n in GLOO_SIZES] + [(c, 1_000_003) for c in GLOO_LARGE]
    for case, n in jobs:
        for dtype in (torch.float32, torch.float64):
            x = make_case(case, n).to(dtype)
            for cut in _splits(n):
                mine = x[:cut] if rank == 0 else x[cut:]
                for q in QS + exact_qs(n):
                    res[(case, n, str(dtype), cut, q)] = par.global_quantile(mine, q)
    torch.save(res, os.path.join(out_dir, f"rank{rank}.pt"))
    dist.barrier()
    dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.fixture(scope="module")
def gloo_results():
    world = 2
    with tempfile.TemporaryDirectory() as d:
        mp.spawn(_gloo_worker, args=(world, _free_port(), d), nprocs=world, join=True)
        yield [torch.load(os.path.join(d, f"rank{r}.pt"), weights_only=False) for r in range(world)]


def test_two_gloo_ranks_match_float64_order_statistics(gloo_results):
    """Uneven shards, an empty shard on either rank, and (case nan) a NaN present on one rank only."""
    r0, r1 = gloo_results
    assert r0.keys() == r1.keys() and len(r0) > 0
    for (case, n, dtype, cut, q), got in r0.items():
        assert bits(got) == bits(r1[(case, n, dtype, cut, q)]), (case, n, dtype, cut, q)  # same on every rank
    for case, n in [(c, n) for c in CASES for n in GLOO_SIZES] + [(c, 1_000_003) for c in GLOO_LARGE]:
        for dtype in (torch.float32, torch.float64):
            x = make_case(case, n).to(dtype)
            for cut in _splits(n):
                check_all_qs(x, lambda q: r0[(case, n, str(dtype), cut, q)])


# ---- device path -------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def engine():
    from amp_extensions_b200.engine import Engine
    return Engine(8, 2, 2, [16], precision="fp16")


@pytest.mark.gpu
@pytest.mark.parametrize("n", SIZES + ((1 << 24) + 3,))
@pytest.mark.parametrize("case", CASES)
def test_device_path_matches_float64_order_statistics(engine, case, n):
    """CUDA fp32 with an engine: simstep_quantile_op.  2^24 + 3 samples are beyond torch.quantile: the sort
    reference with torch's lerp stands in for it."""
    x = make_case(case, n).cuda()
    check_all_qs(x, lambda q: parallel.global_quantile(x, q, engine=engine))
    q1 = parallel.global_quantile(x, 0.9, engine=engine)
    assert bits(q1) == bits(parallel.global_quantile(x, 0.9, engine=engine))


@pytest.mark.gpu
def test_device_path_rejects_q_outside_unit_interval(engine):
    with pytest.raises(ValueError):
        parallel.global_quantile(make_case("uniform", 10).cuda(), 1.5, engine=engine)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ("lognormal6", "bothinf", "nan", "subnormal_max"))
def test_cuda_fp64_takes_the_torch_path(engine, case):
    x = make_case(case, 4097).double().cuda()
    check_all_qs(x, lambda q: parallel.global_quantile(x, q, engine=engine))


def _nccl_worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    device = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=device)
    from amp_extensions_b200 import parallel as par
    from amp_extensions_b200.engine import Engine
    eng = Engine(8, 2, 2, [16], precision="fp16", device=device)
    res = {}
    for case in ("nan", "lognormal6", "zeros90", "bothinf"):
        for n in (3, 4097, 1_000_003):
            x = make_case(case, n)
            for cut in _splits(n):
                mine = (x[:cut] if rank == 0 else x[cut:]).to(device)
                for q in QS + exact_qs(n):
                    res[(case, n, cut, q)] = par.global_quantile(mine, q, engine=eng)
    torch.save(res, os.path.join(out_dir, f"rank{rank}.pt"))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_gpu_device_path_matches_float64_order_statistics():
    """Two NCCL ranks, uneven and empty shards; in case nan the NaN sits on one rank only."""
    world = 2
    with tempfile.TemporaryDirectory() as d:
        mp.spawn(_nccl_worker, args=(world, _free_port(), d), nprocs=world, join=True)
        r0, r1 = [torch.load(os.path.join(d, f"rank{r}.pt"), weights_only=False) for r in range(world)]
    assert r0.keys() == r1.keys() and len(r0) > 0
    for key, got in r0.items():
        assert bits(got) == bits(r1[key]), key
    for case in ("nan", "lognormal6", "zeros90", "bothinf"):
        for n in (3, 4097, 1_000_003):
            x = make_case(case, n)
            for cut in _splits(n):
                check_all_qs(x, lambda q: r0[(case, n, cut, q)])


# ---- simstep_reduce_max_sum: the dataset-maximum threshold -----------------------------------------------------

MAXSUM_SIZES = (0, 1, 31, 33, 1025, 65_536)


def _maxsum_inputs(n):
    g = torch.Generator().manual_seed(n)
    base = torch.randn(n, generator=g) * 3.0
    yield "normal", base
    yield "negative", -base.abs() - 1.0  # the maximum is negative: the -inf start must not leak
    if n == 0:
        return
    for where in sorted({0, n // 2, n - 1}):
        for name, val in (("nan", math.nan), ("posinf", math.inf), ("neginf", -math.inf)):
            x = base.clone()
            x[where] = val
            yield f"{name}@{where}", x
    x = base.clone()
    x[0], x[n - 1] = math.inf, math.nan
    yield "inf_and_nan", x
    if n > 1:
        x = base.clone()
        x[0], x[n - 1] = math.inf, -math.inf
        yield "both_inf", x
    yield "all_neginf", torch.full((n,), -math.inf)


@pytest.mark.gpu
@pytest.mark.parametrize("n", MAXSUM_SIZES)
def test_reduce_max_sum_matches_numpy_float64(engine, n):
    """Maximum bit-exact, NaN-propagating (-inf for no samples); sum within fp64 rounding of the float64 sum."""
    for name, x in _maxsum_inputs(n):
        got = engine.reduce_max_sum(x.cuda()).cpu().tolist()
        xd = x.double().numpy()
        want_max = float(np.max(xd)) if n else -math.inf  # np.max propagates NaN
        want_sum = float(np.sum(xd))
        if math.isnan(want_max):
            assert math.isnan(got[0]), (name, got)
        else:
            assert got[0] == want_max, (name, got[0], want_max)
        if not math.isfinite(want_sum):
            assert (math.isnan(got[1]) and math.isnan(want_sum)) or got[1] == want_sum, (name, got[1], want_sum)
        else:
            assert abs(got[1] - want_sum) <= 4 * n * np.finfo(np.float64).eps * float(np.abs(xd).sum()), name
