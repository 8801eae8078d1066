"""Multi-GPU plumbing: envs shard by index, one process per GPU, full ensemble replica per GPU.

The env step itself needs no data-path collective (every env is independent; SURVEY.md section 8e).
torch.distributed (NCCL on GPUs, gloo in the CPU tests) carries only small reductions:

  * the discrepancy threshold = dataset maximum (reference milo/milo/dynamics.py:145-152) -> all-reduce MAX,
    or, as an extension, a global quantile of the per-row discrepancies via radix-select histogram all-reduces;
  * fit_cost's feature mean (reference milo/milo/linear_cost.py:84-94) -> all-reduce SUM of [D] sums + count;
  * rollout cost / return statistics (reference mjrl/mjrl/algos/batch_reinforce.py:135-141, 288-295);
  * normalisation statistics of a sharded offline dataset (reference milo/milo/datasets.py:23-43).

Every function works un-initialised (world size 1) and on CPU tensors (gloo) as well as CUDA tensors (NCCL).
"""
import math
import struct

import torch
import torch.distributed as dist


def is_dist():
    return dist.is_available() and dist.is_initialized()


def world_size():
    return dist.get_world_size() if is_dist() else 1


def rank():
    return dist.get_rank() if is_dist() else 0


def shard_range(n, rank_=None, world=None):
    """Contiguous env-index range [start, stop) owned by a rank; sizes differ by at most one."""
    r = rank() if rank_ is None else rank_
    w = world_size() if world is None else world
    base, rem = divmod(int(n), w)
    start = r * base + min(r, rem)
    return start, start + base + (1 if r < rem else 0)


def bind_host_to_gpu(device_index):
    """Pin this process to the CPU cores (and thereby the NUMA node) closest to its GPU before any pinned host
    buffer is allocated: with one process per GPU the host<->device copies of all ranks otherwise share whichever
    socket the launcher happened to start them on.  Returns the CPU list, or None when NVML / affinity is not
    available (nothing is changed then)."""
    import os
    try:
        import pynvml
        pynvml.nvmlInit()
        props = torch.cuda.get_device_properties(device_index)
        bus = f"{props.pci_domain_id:08x}:{props.pci_bus_id:02x}:{props.pci_device_id:02x}.0"
        h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [64 * i + b for i, w in enumerate(mask) for b in range(64) if (int(w) >> b) & 1]
        allowed = os.sched_getaffinity(0)
        cpus = sorted(c for c in cpus if c in allowed)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return cpus
    except Exception:
        return None


def _all_reduce(t, op):
    if is_dist():
        dist.all_reduce(t, op=op)
    return t


def all_reduce_max(x):
    """Global maximum of a scalar / tensor (element-wise), NaN-propagating like torch.max."""
    x = torch.as_tensor(x).clone()
    nan = torch.isnan(x).to(x.dtype)
    _all_reduce(nan, dist.ReduceOp.MAX)
    x = torch.nan_to_num(x, nan=-float("inf"))
    _all_reduce(x, dist.ReduceOp.MAX)
    return torch.where(nan > 0, torch.full_like(x, float("nan")), x)


def all_reduce_sum(x):
    return _all_reduce(torch.as_tensor(x).clone(), dist.ReduceOp.SUM)


def global_threshold(ensemble):
    """DynamicsEnsemble.compute_threshold over a dataset sharded across ranks: each rank takes the maximum
    over its own train_dataset on its GPU, one all-reduce(MAX) of a single float makes it global."""
    local = ensemble.dataset_discrepancy_max()
    ensemble.threshold = float(all_reduce_max(local).item())
    return ensemble.threshold


def global_fit_cost(cost, data_pi_local):
    """RBFLinearCost.fit_cost with the rollout rows sharded across ranks: w = global mean phi - phi_e."""
    eng = cost._precise_engine() if hasattr(cost, "_precise_engine") else cost.engine()
    n_local = int(data_pi_local.shape[0])
    if n_local > 0:
        _, psum = eng.rff_features(data_pi_local, want_sum=True)
    else:
        psum = torch.zeros(cost.feature_dim, device=eng.device, dtype=torch.float64)
    packed = torch.cat([psum, torch.tensor([float(n_local)], device=psum.device, dtype=torch.float64)])
    packed = all_reduce_sum(packed)
    phi = (packed[:-1] / packed[-1].clamp_min(1.0)).float().cpu()
    cost.w = phi - cost.phi_e
    return cost.w


def global_mean(sum_local, count_local):
    """Mean of a quantity whose per-rank sums and counts are given (fp64)."""
    packed = torch.cat([torch.as_tensor(sum_local, dtype=torch.float64).reshape(-1),
                        torch.as_tensor([float(count_local)], dtype=torch.float64).to(torch.as_tensor(sum_local).device)])
    packed = all_reduce_sum(packed)
    return packed[:-1] / packed[-1].clamp_min(1.0)


def global_transformations(states_local, actions_local, next_states_local):
    """AmpDataset.get_transformations (datasets.py:23-43) over an offline dataset whose rows are sharded across
    ranks: two passes, each one all-reduce(SUM) of the per-rank column sums (fp64) — first the means, then the mean
    absolute deviations around the GLOBAL means.  Returns the reference's tuple (state_mean, state_scale,
    action_mean, action_scale, diff_mean, diff_scale) as fp32 tensors, identical on every rank.  Host-side
    statistics, computed once when the ensemble is built (the reference does the same on the host)."""
    parts = [states_local.double(), actions_local.double(), (next_states_local - states_local).double()]
    n_local = float(states_local.shape[0])
    widths = [p.shape[1] for p in parts]
    packed = torch.cat([p.sum(dim=0) for p in parts] + [torch.tensor([n_local], dtype=torch.float64)])
    packed = all_reduce_sum(packed)
    n = packed[-1].clamp_min(1.0)
    means = [m.float() for m in torch.split(packed[:-1] / n, widths)]
    dev = torch.cat([(p.float() - m).abs().double().sum(dim=0) for p, m in zip(parts, means)])
    dev = all_reduce_sum(dev)
    scales = [(d / n).float() + 1e-8 for d in torch.split(dev, widths)]
    return (means[0], scales[0], means[1], scales[1], means[2], scales[2])


def rollout_stats(cost, ipm, bonus, done, num_steps):
    """Global rollout statistics of one batch of env-steps (batch_reinforce.py:135-141, 288-295):
    sums / extrema of reward = -cost, int = -bonus, ext = -ipm, finished episodes and their lengths."""
    f = torch.float64
    done_b = done.to(torch.bool)
    n = torch.tensor(float(cost.numel()), device=cost.device, dtype=f)
    sums = torch.stack([(-cost).to(f).sum(), ((-cost).to(f) ** 2).sum(), (-bonus).to(f).sum(), (-ipm).to(f).sum(),
                        done_b.to(f).sum(), (num_steps.to(f) * done_b.to(f)).sum(), n])
    big = float("inf")
    mx = torch.stack([(-cost).to(f).max() if cost.numel() else torch.tensor(-big, device=cost.device, dtype=f),
                      cost.to(f).max() if cost.numel() else torch.tensor(-big, device=cost.device, dtype=f)])
    sums = all_reduce_sum(sums)
    mx = all_reduce_max(mx)
    count = sums[6].clamp_min(1.0)
    mean = sums[0] / count
    var = (sums[1] / count - mean * mean).clamp_min(0.0)
    return {
        "n": int(sums[6].item()), "reward_mean": float(mean), "reward_std": float(var.sqrt()),
        "reward_max": float(mx[0]), "reward_min": float(-mx[1]), "int": float(sums[2]), "ext": float(sums[3]),
        "episodes_done": int(sums[4].item()),
        "ep_len_mean": float(sums[5] / sums[4].clamp_min(1.0)),
    }


def _global_quantile_device(x32, q, engine):
    """Device-resident variant of the radix selection (simstep_quantile_op): the prefixes, ranks and result live in
    device memory, so the call issues 3 all-reduces of the counts and synchronises with the host ONCE, for the
    result."""
    qstate = torch.zeros(12, device=x32.device, dtype=torch.float64)
    qstate[0] = q
    counts = torch.empty(2 * engine.QUANTILE_BINS + 1, device=x32.device, dtype=torch.int64)
    for _ in range(3):  # 12 + 12 + 8 key bits
        engine.quantile_op(engine.QOP_HIST, x32, qstate=qstate, counts=counts)
        _all_reduce(counts, dist.ReduceOp.SUM)
        engine.quantile_op(engine.QOP_SELECT, None, qstate=qstate, counts=counts)
    return float(qstate[1].item())


# dtype -> (integer view, key bits, digit widths of the passes, struct formats of the integer and the float)
_KEYS = {torch.float32: (torch.int32, 32, (12, 12, 8), "<i", "<f"),
         torch.float64: (torch.int64, 64, (16, 16, 16, 16), "<q", "<d")}


def _order_stats(x, q):
    """Torch path of global_quantile: (v0, v1, w) with v0, v1 the order statistics k0 = floor(q (n - 1)) and
    min(k0 + 1, n - 1) of the union of every rank's x (fp32 or fp64) and w = q (n - 1) - k0, or None when there are no
    samples or any NaN.  Radix selection on the signed order-preserving key of the bit pattern,
    key = s ^ ((s >> (B - 1)) & (2^(B-1) - 1)); digit d of a pass counts the samples that share the prefix fixed so
    far (top digit offset by 2^(w-1) to make it unsigned); one all-reduce of the counts per pass."""
    view, nbits, widths, ifmt, ffmt = _KEYS[x.dtype]
    nan = torch.isnan(x)
    s = x[~nan].view(view).to(torch.int64)
    key = s ^ ((s >> (nbits - 1)) & ((1 << (nbits - 1)) - 1))
    keys, below, prefix = [key, key], [0, 0], [0, 0]
    fixed = 0
    for p, w in enumerate(widths):
        shift = nbits - fixed - w
        same = prefix[0] == prefix[1]  # both order statistics still share their prefix: one histogram serves both
        digits = [((k >> shift) & ((1 << w) - 1)) ^ ((1 << (w - 1)) if p == 0 else 0) for k in keys[:1 if same else 2]]
        hists = [torch.bincount(d, minlength=1 << w) for d in digits]
        head = [nan.sum().reshape(1)] if p == 0 else []
        packed = all_reduce_sum(torch.cat(hists + head))
        if p == 0:
            n_nan = int(packed[-1])
            n = int(packed[:-1].sum()) + n_nan
            if n_nan or n == 0:
                return None
            pos = q * (n - 1)
            k0 = math.floor(pos)
            ks, wt = (k0, min(k0 + 1, n - 1)), pos - k0
        for i in range(2):
            j = 0 if same else i
            cum = torch.cumsum(packed[j << w:(j + 1) << w], 0) + below[i]
            b = int(torch.searchsorted(cum, torch.tensor([ks[i]], device=cum.device), right=True))
            below[i] = int(cum[b - 1]) if b > 0 else below[i]
            prefix[i] = (prefix[i] << w) | b
            keys.append(keys[j][digits[j] == b])
        keys = keys[2:]
        fixed += w

    def value(ukey):
        key = ukey - (1 << (nbits - 1))
        s = key ^ ((key >> (nbits - 1)) & ((1 << (nbits - 1)) - 1))
        return struct.unpack(ffmt, struct.pack(ifmt, s))[0]

    return value(prefix[0]), value(prefix[1]), wt


def global_quantile(x_local, q, engine=None):
    """q-quantile of the union of every rank's x_local, without gathering the samples: the linear interpolation
    between the order statistics k0 = floor(q (n - 1)) and k0 + 1 of torch.quantile, used for
    threshold_mode='quantile' (an extension over the reference's dataset maximum).

    The order statistics are exact: radix selection on the order-preserving integer key of the bit pattern, one
    all-reduce of a histogram of the next key digit per pass (fp32: 12 + 12 + 8 bits, fp64: 4 x 16 bits; other dtypes
    go through fp64).  Semantics:
      * any NaN in the union of the samples, or no samples at all, gives NaN; q outside [0, 1] raises ValueError;
      * w = q (n - 1) - k0 == 0 gives sorted[k0] exactly.  This deliberately differs from torch.quantile where it
        returns NaN for lerp(inf, inf, 0), e.g. at q = 1 when the maximum is +inf;
      * otherwise torch.lerp's formula in fp64, v0 + w (v1 - v0) for w < 0.5 and v1 - (v1 - v0)(1 - w) above.
    With `engine` and a CUDA fp32 vector everything but the final read stays on the device (_global_quantile_device);
    other tensors (CPU ones in the gloo tests, CUDA fp64) take the torch path."""
    q = float(q)
    if not 0.0 <= q <= 1.0:
        raise ValueError(f"quantile q must be in [0, 1], got {q}")
    xt = torch.as_tensor(x_local).reshape(-1)
    if engine is not None and xt.is_cuda and xt.dtype == torch.float32:
        return _global_quantile_device(xt.contiguous(), q, engine)
    if xt.dtype not in _KEYS:
        xt = xt.to(torch.float64)
    stats = _order_stats(xt.contiguous(), q)
    if stats is None:
        return float("nan")
    v0, v1, w = stats
    if w == 0.0:
        return v0
    f64 = torch.float64
    return float(torch.lerp(torch.tensor(v0, dtype=f64), torch.tensor(v1, dtype=f64), w))
