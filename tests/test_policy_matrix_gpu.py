"""The rollout policy's forward (policy_act_kernel, csrc/policy.cuh) and the on-device NPG step (simstep_npg_*,
csrc/npg.cuh, csrc/npg_api.inc) at every policy shape, row count and mask their launch code dispatches on, against the
float64 oracle oracle/npg_oracle.py on the fp32 parameters (Policy.mean, vpg_grad, hvp, npg_step).

Gradient and Fisher-vector sums are bounded per tensor - each layer's W, each layer's b, log_std - relative to that
tensor's largest entry, so one wrong bias column or log_std entry fails where a relative L2 over the whole vector would
not.  A relu unit whose pre-activation sits within the fp32 rounding band of zero flips its mask between kernel and
oracle, so relu cases draw their rows from those whose every hidden pre-activation clears MASK_MARGIN of the layer's
largest (select_rows) instead of loosening the bound.

Rows masked out by `valid` must not matter: the sums with NaN / +-Inf in a masked row's observation, action and
advantage are bit-identical to the sums with that row zero-filled.  A policy with no valid row (or no row) leaves the
parameters unchanged; the oracle's means are NaN there, so that is the defined device behaviour.

The CPU section restates npg_init / npg_plan and simstep_load_policy's shared-memory check and checks that the case
table reaches every branch; the GPU section checks the restatement's accept / refuse decisions against the library.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import npg_oracle as no

# Per-tensor bounds relative to the tensor's largest entry, about twice the worst error measured on one NVIDIA B200
# (power limit 1000 W) over every case, row count and mask of test_policy_mean_matches_the_oracle and
# test_gradient_and_fvp_match_the_oracle.  Worst: policy mean 1.76e-6 (obs512); gradient weight 1.33e-6 (relu64), bias
# 1.21e-6 (relu64), log_std 1.69e-6 (relu_tf); Fisher-vector weight 1.37e-6 and bias 1.13e-6 (obs512).  The
# Fisher-vector log_std entries are the fp64 closed form count * h(s) * v, 7.2e-15 (relu64).
REL = {"mean": 4e-6,
       "grad": {"weight": 3e-6, "bias": 2.5e-6, "log_std": 3.5e-6},
       "fvp": {"weight": 3e-6, "bias": 2.5e-6, "log_std": 2e-14}}
UPDATE_REL = 1e-3      # a whole update (test_npg_gpu.py's budget): relative L2 of theta_new - theta, and the scalars
MASK_MARGIN = 1e-4     # relu: |pre-activation| > MASK_MARGIN * the layer's largest, so fp32 error cannot flip a mask
MIN_LOG_STD = -3.0

# the launch code's constants (csrc/npg.cuh, csrc/policy.cuh, npg_api.inc, policy_api.inc)
NPG_THREADS, NPG_MAX_ITEMS, NPG_EXTRA = 512, 3, 4
NPG_MAX_BLOCKS = NPG_THREADS * NPG_MAX_ITEMS
SMEM_LIMIT = 200 * 1024
POLICY_MAX_LAYERS, POLICY_MAX_WIDTH, POLICY_MAX_IN, POLICY_WARPS, POLICY_ENVS = 4, 128, 512, 4, 4
N_SM = 148             # B200: the row kernels' grid is min(tiles, SMs)

# id, layer sizes, nonlinearity, transforms, the branch the row exists for
CASES = [
    dict(id="polA", sizes=[226, 32, 32, 28], act="tanh", covers="the MILO shape: R = 64, 591 blocks (two per thread)"),
    dict(id="relu64", sizes=[226, 64, 64, 28], act="relu", covers="mjrl's default widths: R = 32, three blocks per thread"),
    dict(id="linear", sizes=[226, 28], act="tanh", covers="L = 1: no hidden layer, no activation cache"),
    dict(id="four_layer", sizes=[20, 24, 24, 24, 5], act="tanh", covers="L = 4 at R = 64"),
    dict(id="in3mod4", sizes=[11, 19, 6], act="tanh",
         covers="in + 1 = 0 mod 4 (the bias column ends a quad); outputs 3 and 2 mod 4"),
    # width1's 11-parameter Fisher has condition number 1.2e3 at damping 1e-4: a 1e-6 relative change of its sums
    # moves the CG solution by 2e-3, so a whole update is held to 1e-2 (measured 4.9e-3), its sums per entry above
    dict(id="width1", sizes=[7, 1, 1], act="tanh", covers="width 1: one unit in a quad, one in a 32-wide pad",
         update_rel=1e-2),
    dict(id="obs1", sizes=[1, 5, 3], act="tanh", covers="obs_dim = 1: the bias column shares the only k-quad"),
    dict(id="act128", sizes=[16, 128], act="tanh", covers="act_dim = 128: four lane passes in the policy kernel"),
    dict(id="act33", sizes=[24, 40, 33], act="tanh", covers="act_dim = 33: a second lane pass of one unit"),
    dict(id="obs512", sizes=[512, 32, 4], act="tanh",
         covers="obs_dim = kPolicyMaxIn: 512-wide activation buffers, R = 32, three blocks per thread"),
    dict(id="blocks1536", sizes=[160, 125, 28], act="tanh", covers="exactly kNpgMaxBlocks gradient blocks"),
    dict(id="relu_tf", sizes=[40, 64, 48, 33, 12], act="relu", transform=True,
         covers="relu with all four transforms and a zero in_scale column, L = 4 at R = 32"),
]
REFUSED = [
    dict(id="blocks1537", sizes=[184, 128, 1], act="tanh", covers="one block over kNpgMaxBlocks; shared memory fits"),
    dict(id="smem_only", sizes=[8, 96, 96, 96, 1], act="tanh", covers="1297 blocks; even R = 32 overflows shared memory"),
]
CASE = {c["id"]: c for c in CASES + REFUSED}
IDS = [c["id"] for c in CASES]
MASKS = ["none", "valid", "idx", "idx_valid"]
ZERO_SCALE_COL = 3     # relu_tf: in_scale 0 there (a constant observation feature in mjrl's transforms)


# ---------------------------------------------------------------------------------------------------
# the launch code restated (CPU)


def rup(x, m):
    return (x + m - 1) // m * m


def npg_stride(w):
    return (w + 7) // 8 * 8 + 4


def policy_geometry(sizes):
    """simstep_load_policy's PolicyConst: per layer (in, out, out_pad), pack floats and policy_smem_bytes."""
    ins, outs = sizes[:-1], sizes[1:]
    pads = [rup(o, 32) for o in outs]
    pack = sum(i * p + p for i, p in zip(ins, pads))
    width = max(sizes[0], POLICY_MAX_WIDTH)
    smem = (pack + POLICY_WARPS * 2 * width * POLICY_ENVS) * 4
    ok = (1 <= len(outs) <= POLICY_MAX_LAYERS and 1 <= sizes[0] <= POLICY_MAX_IN
          and all(1 <= o <= POLICY_MAX_WIDTH for o in outs) and smem <= SMEM_LIMIT)
    return dict(ins=ins, outs=outs, pads=pads, pack=pack, width=width, smem=smem, ok=ok)


def npg_smem(sizes, R):
    """npg_plan: bytes of the row kernels' shared memory at R rows per tile."""
    g = policy_geometry(sizes)
    ins, outs = g["ins"], g["outs"]
    off = rup(g["pack"], 4)
    sa = [npg_stride(i + 1) for i in ins]
    sd = [npg_stride(o) for o in outs]
    off += R * sum(sa)            # a_l
    off += R * sum(sa[1:])        # da_l, l >= 1
    off += R * sd[-1]             # DIAG: the old parameters' output layer
    off += R * sum(sd)            # delta_l
    off += R * npg_stride(outs[-1] + NPG_EXTRA)
    return off * 4


def npg_geometry(sizes):
    """npg_init's decisions: gradient blocks, k-quads, items per thread, R, cache width, and which refusal applies."""
    g = policy_geometry(sizes)
    kq = [(i + 1 + 3) // 4 for i in g["ins"]]
    blocks = sum(((o + 3) // 4) * k for o, k in zip(g["outs"], kq))
    R = 64 if npg_smem(sizes, 64) <= SMEM_LIMIT else 32
    refused = None
    if blocks > NPG_MAX_BLOCKS:
        refused = "blocks"
    elif npg_smem(sizes, 32) > SMEM_LIMIT:
        refused = "smem"
    return dict(g, kq=kq, blocks=blocks, items=(blocks + NPG_THREADS - 1) // NPG_THREADS, R=R, refused=refused,
                cache_w=sum(g["ins"][1:]), n_params=sum(o * i + o for i, o in zip(g["ins"], g["outs"])) + sizes[-1])


def row_counts(R):
    """1, R - 1, R + 1 and 2 * SMs * R + 17 (every CTA walks two or three tiles, the last one ragged)."""
    return [1, R - 1, R + 1, 2 * N_SM * R + 17]


def npg_branches(c):
    """The npg_init / row kernel / policy kernel branches case c takes at its row counts and masks."""
    q, b = npg_geometry(c["sizes"]), set()
    if q["refused"]:
        b.add(("refused", q["refused"]))
        if q["refused"] == "blocks" and npg_smem(c["sizes"], 32) <= SMEM_LIMIT:
            b.add(("refused by the block count alone",))
        if q["refused"] == "smem" and q["blocks"] <= NPG_MAX_BLOCKS:
            b.add(("refused by shared memory alone",))
        if q["blocks"] == NPG_MAX_BLOCKS + 1:
            b.add(("blocks", "kNpgMaxBlocks + 1"))
        return b
    b.add(("R", q["R"]))
    b.add(("items per thread", q["items"]))
    if q["blocks"] == NPG_MAX_BLOCKS:
        b.add(("blocks", "kNpgMaxBlocks"))
    L = len(q["outs"])
    b.add(("layers", L))
    b.add(("cache", "none" if q["cache_w"] == 0 else "hidden activations"))
    for i in q["ins"]:
        b.add(("in mod 4", i % 4))        # 3: the bias column ends a quad; 0: it starts one alone
    for o in q["outs"]:
        b.add(("out mod 4", o % 4))
    b.add(("policy lane passes", max(p // 32 for p in q["pads"])))
    b.add(("act_dim > 32", c["sizes"][-1] > 32))
    b.add(("policy buffers", "obs_dim wide" if c["sizes"][0] > POLICY_MAX_WIDTH else "128 wide"))
    if c["sizes"][0] == POLICY_MAX_IN:
        b.add(("obs_dim", "kPolicyMaxIn"))
    if min(c["sizes"]) == 1:
        b.add(("a width of 1",))
    b.add(("activation", c["act"]))
    if c.get("transform"):
        b.add(("transforms", "with a zero in_scale column"))
    for n in row_counts(q["R"]):
        tiles = (n + q["R"] - 1) // q["R"]
        b.add(("rows", "one" if n == 1 else "ragged last tile" if n % q["R"] else "whole tiles"))
        b.add(("grid", "fewer tiles than SMs" if tiles < N_SM else "several tiles per CTA" if tiles > 2 * N_SM
               else "one or two tiles per CTA"))
    b |= {("mask", m) for m in MASKS}
    return b


# ---------------------------------------------------------------------------------------------------
# case data (CPU)

_cache = {}


def hidden_pre(pol, theta, obs):
    """Pre-activations of every hidden layer, float64 (Policy.mean's arithmetic)."""
    ws, bs, _ = pol.unflatten(theta)
    act = torch.relu if pol.nonlinearity == "relu" else torch.tanh
    h = (torch.as_tensor(obs, dtype=torch.float64) - pol.in_shift) / (pol.in_scale + 1e-8)
    pres = []
    for w, b in zip(ws[:-1], bs[:-1]):
        pres.append(h @ w.T + b)
        h = act(pres[-1])
    return pres


def select_rows(pol, theta, obs):
    """relu: the rows whose every hidden pre-activation clears MASK_MARGIN of the layer's largest |pre-activation|."""
    if pol.nonlinearity != "relu" or len(pol.sizes) == 2:
        return obs
    ok = torch.ones(obs.shape[0], dtype=torch.bool)
    for p in hidden_pre(pol, theta, obs):
        ok &= (p.abs() > MASK_MARGIN * float(p.abs().max())).all(dim=1)
    return obs[ok]


def case_data(cid):
    """Policy (oracle object, fp32 theta, engine.load_policy kwargs) and rows of a case (seeded, cached)."""
    if cid in _cache:
        return _cache[cid]
    c = dict(CASE[cid])
    seed = 400 + list(CASE).index(cid)
    g = torch.Generator().manual_seed(seed)
    sizes = c["sizes"]
    obs_dim, A = sizes[0], sizes[-1]
    ws = [torch.randn(o, i, generator=g) * (1.2 / i ** 0.5) for i, o in zip(sizes[:-1], sizes[1:])]
    bs = [torch.randn(o, generator=g) * 0.2 for o in sizes[1:]]
    ls = -0.5 + 0.2 * torch.randn(A, generator=g)
    tf = {}
    if c.get("transform"):
        tf = dict(in_shift=0.5 * torch.randn(obs_dim, generator=g), in_scale=0.5 + torch.rand(obs_dim, generator=g),
                  out_shift=0.3 * torch.randn(A, generator=g), out_scale=0.5 + torch.rand(A, generator=g))
        tf["in_shift"][ZERO_SCALE_COL] = 0.0
        tf["in_scale"][ZERO_SCALE_COL] = 0.0
    pol = no.Policy(sizes, c["act"], **{k: v.double() for k, v in tf.items()}, min_log_std=MIN_LOG_STD)
    theta = pol.flatten(ws, bs, ls).float()
    q = npg_geometry(sizes)
    n_max = row_counts(q["R"])[-1] if not q["refused"] else 1024
    obs = torch.randn(2 * n_max, obs_dim, generator=g)
    if tf:
        obs = obs * tf["in_scale"] + tf["in_shift"]
        # in_scale 0: the feature divides by fp32(0 + 1e-8) on the device and by 1e-8 in the oracle (6e-9 apart);
        # observations of order 1e-9 keep the normalised value of order 0.1
        obs[:, ZERO_SCALE_COL] = 1e-9 * torch.randn(obs.shape[0], generator=g)
    obs = select_rows(pol, theta.double(), obs)
    assert obs.shape[0] >= n_max, (cid, obs.shape[0], n_max)
    obs = obs[:n_max].contiguous()
    mu = pol.mean(theta.double(), obs).float()
    z = torch.randn(n_max, A, generator=g)
    act = (mu + torch.exp(ls) * z).contiguous()
    # advantages that follow the actions (a policy gradient with signal, not only sampling noise), as multiples of
    # 1/64 with |adv| <= 4: every fp32 partial sum of up to 2^17 of them is exact
    u = torch.randn(A, generator=g)
    adv = (z @ u) / float(u.norm()) + 0.5 * torch.randn(n_max, generator=g)
    adv = (adv * 64).round().clamp(-256, 256) / 64
    kw = dict(weights=ws, biases=bs, nonlinearity=c["act"], log_std=ls, **tf)
    c.update(pol=pol, theta=theta, kw=kw, obs=obs, act=act, adv=adv, q=q, seed=seed)
    _cache[cid] = c
    return c


def masks(n, seed):
    """{mask name: (valid uint8 [n] or None, Fisher indices int64 or None)}: a random 70 % valid mask and indices with
    duplicates."""
    g = torch.Generator().manual_seed(seed)
    valid = (torch.rand(n, generator=g) < 0.7).to(torch.uint8)
    idx = torch.randint(0, n, (n // 2 + 1,), generator=g)
    idx = torch.cat([idx, idx[:1]])   # at least one duplicate
    return {"none": (None, None), "valid": (valid, None), "idx": (None, idx), "idx_valid": (valid, idx)}


def parts(pol, v):
    """{(kind, layer): tensor} of a flat parameter-sized vector."""
    ws, bs, ls = pol.unflatten(torch.as_tensor(v, dtype=torch.float64))
    d = {("weight", l): w for l, w in enumerate(ws)}
    d.update({("bias", l): b for l, b in enumerate(bs)})
    d[("log_std", 0)] = ls
    return d


def rel_to_max(x, ref):
    x, ref = np.asarray(x, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    return float(np.abs(x - ref).max() / max(np.abs(ref).max(), 1e-30))


def check_parts(pol, got, ref, bounds, tag, worst):
    """Per-tensor bound relative to the tensor's largest entry; records the worst error per kind in `worst`."""
    pg, pr = parts(pol, got), parts(pol, ref)
    for key, r in pr.items():
        e = rel_to_max(pg[key], r)
        worst[key[0]] = max(worst.get(key[0], 0.0), e)
        assert e <= bounds[key[0]], (tag, key, e)


def rel_l2(x, ref):
    x, ref = torch.as_tensor(x, dtype=torch.float64).cpu(), torch.as_tensor(ref, dtype=torch.float64).cpu()
    return float(torch.linalg.norm(x - ref) / torch.linalg.norm(ref))


# ---------------------------------------------------------------------------------------------------
# GPU: engines


def engine():
    from tests import helpers as H
    from tests.test_parity_gpu import make_engine
    return make_engine(H.tiny_case("tiny_dense"), "fp16")


def load(eng, c, theta=None):
    kw = c["kw"]
    eng.load_policy(kw["weights"], kw["biases"], kw["nonlinearity"], kw.get("in_shift"), kw.get("in_scale"),
                    kw.get("out_shift"), kw.get("out_scale"), kw["log_std"])
    if theta is not None:
        eng.npg_init(MIN_LOG_STD)
        eng.npg_params(theta.cuda())


def host_policy(c, theta):
    from tests.test_npg_gpu import _HostPolicy
    host = _HostPolicy(c["kw"], theta)
    ws, bs, ls = c["pol"].unflatten(theta.double())
    for layer, w, b in zip(host.model.fc_layers, ws, bs):
        layer.weight.data, layer.bias.data = w.float().clone(), b.float().clone()
    host.log_std = ls.float().clone()
    host.min_log_std = MIN_LOG_STD
    return host


# ---------------------------------------------------------------------------------------------------
# GPU: the policy forward


@pytest.mark.gpu
@pytest.mark.parametrize("cid", IDS)
def test_policy_mean_matches_the_oracle(cid):
    """policy_act's mean against Policy.mean per entry; the noisy action is fmaf(std, noise, mean) within an ulp; the
    evaluation action is the mean; mean-only and action-only calls return the combined call's values bit for bit."""
    from amp_extensions_b200 import engine as E
    c = case_data(cid)
    eng = engine()
    load(eng, c)
    pol, theta = c["pol"], c["theta"].double()
    std = torch.exp(c["kw"]["log_std"].double()).float()
    g = torch.Generator().manual_seed(c["seed"])
    worst = 0.0
    for n in row_counts(c["q"]["R"]):
        obs = c["obs"][:n]
        o = obs.cuda()
        noise = torch.randn(n, pol.sizes[-1], generator=g)
        act, mean = eng.policy_act(o, noise.cuda())
        ref = pol.mean(theta, obs)
        e = rel_to_max(mean.cpu(), ref)
        worst = max(worst, e)
        assert e <= REL["mean"], (cid, n, e)
        m = mean.cpu()
        want = (std.double() * noise.double() + m.double()).float()
        assert (torch.abs(act.cpu() - want) <= torch.from_numpy(np.spacing(np.abs(want.numpy())))).all(), (cid, n)
        act_eval, mean_eval = eng.policy_act(o)
        assert torch.equal(act_eval, mean) and torch.equal(mean_eval, mean)
        act_only, none = eng.policy_act(o, noise.cuda(), want_mean=False)
        assert none is None and torch.equal(act_only, act)
        mean_only = torch.full_like(mean, float("nan"))
        eng._check(eng.lib.simstep_policy_act(eng._h, E._ptr(o), E._ptr(noise.cuda()), n, C.c_void_p(0),
                                              E._ptr(mean_only), E._stream(eng.device)))
        assert torch.equal(mean_only, mean)
    print(f"policy mean worst {cid}: {worst:.2e}")


# ---------------------------------------------------------------------------------------------------
# GPU: gradient and Fisher-vector sums


def oracle_sums(c, obs, act, adv, valid, idx, v):
    """Float64 (gradient sum, rows, advantage sum, Fisher-vector sum, Fisher rows) of the rows the masks keep."""
    pol, theta = c["pol"], c["theta"].double()
    keep = torch.ones(obs.shape[0], dtype=torch.bool) if valid is None else valid.bool()
    n = int(keep.sum())
    grad = no.vpg_grad(pol, theta, obs[keep], act[keep], adv[keep]) * n if n else torch.zeros(pol.n_params, dtype=torch.float64)
    fi = torch.arange(obs.shape[0]) if idx is None else idx
    fi = fi[keep[fi]]
    nf = len(fi)
    fvp = no.hvp(pol, theta, obs[fi], v) * nf if nf else torch.zeros(pol.n_params, dtype=torch.float64)
    return grad, n, float(adv.double()[keep].sum()), fvp, nf


@pytest.mark.gpu
@pytest.mark.parametrize("cid", IDS)
def test_gradient_and_fvp_match_the_oracle(cid):
    """npg_grad and npg_prepare + npg_fvp at every row count and mask against vpg_grad / hvp, per tensor; the row-count
    and advantage-sum columns exactly; a repeated call bit for bit."""
    c = case_data(cid)
    eng = engine()
    pol = c["pol"]
    load(eng, c, c["theta"])
    P = pol.n_params
    v = torch.randn(P, generator=torch.Generator().manual_seed(c["seed"]), dtype=torch.float64)
    vd = v.cuda()
    worst = {"grad": {}, "fvp": {}}
    for n in row_counts(c["q"]["R"]):
        obs, act, adv = c["obs"][:n], c["act"][:n], c["adv"][:n]
        o, a, d = obs.cuda(), act.cuda(), adv.cuda()
        for mname, (valid, idx) in masks(n, c["seed"] + n).items():
            vl = None if valid is None else valid.cuda()
            ix = None if idx is None else idx.cuda()
            tag = (cid, n, mname)
            gs = eng.npg_grad(o, a, d, vl).cpu()
            eng.npg_prepare(o, ix)
            fs = eng.npg_fvp(o, vl, ix, v=vd).cpu()
            assert torch.equal(eng.npg_grad(o, a, d, vl).cpu(), gs), tag
            assert torch.equal(eng.npg_fvp(o, vl, ix, v=vd).cpu(), fs), tag
            grad, rows, adv_sum, fvp, frows = oracle_sums(c, obs, act, adv, valid, idx, v)
            assert float(gs[P]) == rows and float(gs[P + 1]) == adv_sum, (tag, float(gs[P]), rows, float(gs[P + 1]), adv_sum)
            assert float(fs[P]) == frows and float(fs[P + 1]) == 0.0, (tag, float(fs[P]), frows)
            if rows:
                check_parts(pol, gs[:P], grad, REL["grad"], tag + ("grad",), worst["grad"])
            else:
                assert not gs[:P].any(), tag
            if frows:
                check_parts(pol, fs[:P], fvp, REL["fvp"], tag + ("fvp",), worst["fvp"])
            else:
                assert not fs[:P].any(), tag
    print(f"worst per tensor {cid}:", {k: {kk: f"{vv:.2e}" for kk, vv in w.items()} for k, w in worst.items()})


def poison(x, valid):
    """x with every masked-out row filled with NaN, +Inf, -Inf in turn."""
    x = x.clone()
    bad = torch.nonzero(valid == 0).flatten()
    vals = torch.tensor([float("nan"), float("inf"), -float("inf")])
    fill = vals[torch.arange(len(bad)) % 3]
    x[bad] = fill.view(-1, *([1] * (x.dim() - 1))).expand(-1, *x.shape[1:])
    return x


@pytest.mark.gpu
@pytest.mark.parametrize("cid", IDS)
def test_masked_rows_do_not_matter(cid):
    """Gradient and Fisher-vector sums with NaN / +-Inf in the masked rows' observations, actions and advantages are
    bit-identical to the sums with those rows zero-filled, with and without Fisher indices."""
    c = case_data(cid)
    eng = engine()
    load(eng, c, c["theta"])
    P = c["pol"].n_params
    vd = torch.randn(P, generator=torch.Generator().manual_seed(c["seed"]), dtype=torch.float64).cuda()
    for n in row_counts(c["q"]["R"])[2:]:
        ms = masks(n, c["seed"] + n)
        for mname in ("valid", "idx_valid"):
            valid, idx = ms[mname]
            vl, ix = valid.cuda(), None if idx is None else idx.cuda()
            out = []
            for fill in ("zero", "nonfinite"):
                rows = [c["obs"][:n], c["act"][:n], c["adv"][:n]]
                if fill == "zero":
                    rows = [t * valid.view(-1, *([1] * (t.dim() - 1))).float() for t in rows]
                else:
                    rows = [poison(t, valid) for t in rows]
                o, a, d = (t.contiguous().cuda() for t in rows)
                gs = eng.npg_grad(o, a, d, vl)
                eng.npg_prepare(o, ix)
                fs = eng.npg_fvp(o, vl, ix, v=vd)
                out.append((gs.cpu(), fs.cpu()))
            tag = (cid, n, mname)
            assert bool(torch.isfinite(out[1][0]).all()), (tag, "gradient sums not finite")
            assert bool(torch.isfinite(out[1][1]).all()), (tag, "Fisher-vector sums not finite")
            assert torch.equal(out[0][0], out[1][0]) and torch.equal(out[0][1], out[1][1]), tag


# ---------------------------------------------------------------------------------------------------
# GPU: whole updates


UPDATE_ROWS = 6000


@pytest.mark.gpu
@pytest.mark.parametrize("cid", IDS)
def test_no_valid_row_leaves_the_parameters_unchanged(cid):
    """Every row masked out (and those rows non-finite), or no row at all: DeviceNPG.update writes back exactly the
    parameters it started from and returns finite scalars (the oracle's means are NaN there)."""
    from amp_extensions_b200.npg import DeviceNPG
    c = case_data(cid)
    n = c["q"]["R"] + 1
    theta = c["theta"]
    npg = DeviceNPG(engine(), host_policy(c, theta))
    valid = torch.zeros(n, dtype=torch.uint8)
    rows = [poison(t[:n], valid).cuda() for t in (c["obs"], c["act"], c["adv"])]
    for label, (o, a, d, vl) in (("all masked", (rows[0], rows[1], rows[2], valid.cuda())),
                                 ("no rows", (rows[0][:0].contiguous(), rows[1][:0].contiguous(),
                                              rows[2][:0].contiguous(), None))):
        out = npg.update((o, a), d, vl)
        assert torch.equal(npg.params().cpu(), theta), (cid, label)
        for k, x in out.items():
            assert bool(torch.isfinite(x).all()), (cid, label, k, x)
        mean = npg.eng.policy_act(c["obs"][:n].cuda())[1].cpu()
        fresh = engine()
        load(fresh, c)
        assert torch.equal(mean, fresh.policy_act(c["obs"][:n].cuda())[1].cpu()), (cid, label)


@pytest.mark.gpu
@pytest.mark.parametrize("cid,clamp", [(cid, False) for cid in IDS] + [("act33", True)])
def test_two_updates_match_chained_oracle_steps(cid, clamp):
    """Two DeviceNPG.update calls (valid mask and HVP subsample) against two chained npg_step calls, each on its own
    previous parameters; the second step only matches if old_pack / old_std were refreshed between the steps.  After
    them, policy_act on the updated handle equals policy_act of a fresh load of npg_params() bit for bit (pack_of at
    every ragged out_pad), and Policy.mean at those parameters per entry.  clamp: log_std starts just above
    min_log_std so the clamp binds."""
    from amp_extensions_b200.npg import DeviceNPG
    c = case_data(cid)
    pol = c["pol"]
    budget = c.get("update_rel", UPDATE_REL)
    n = UPDATE_ROWS
    obs, act = c["obs"][:n], c["act"][:n]
    adv = (c["adv"][:n] - c["adv"][:n].mean()) / c["adv"][:n].std()   # whitened, as the reference's caller does
    theta = c["theta"].clone()
    ls0 = pol.n_params - pol.sizes[-1]
    if clamp:
        theta[ls0:] = MIN_LOG_STD + 1e-4
    g = torch.Generator().manual_seed(c["seed"] + 1)
    valid = (torch.rand(n, generator=g) < 0.8).to(torch.uint8)
    frac = 0.5
    eng = engine()
    npg = DeviceNPG(eng, host_policy(c, theta), hvp_sample_frac=frac, seed=c["seed"])
    gen = torch.Generator(device="cuda")
    gen.manual_seed(c["seed"])
    ref_theta = theta.double()
    o, a, d, vl = obs.cuda(), act.cuda(), adv.cuda(), valid.cuda()
    for step in range(2):
        # the rows DeviceNPG draws: the same generator, the same call
        idx = torch.randint(0, n, (int(frac * n),), device="cuda", generator=gen, dtype=torch.int64).cpu()
        out = {k: float(x) for k, x in npg.update((o, a), d, vl).items()}
        new_ref, ref = no.npg_step(pol, ref_theta, obs, act, adv, valid=valid, fisher_idx=idx, cg_iters=10, damping=1e-4)
        got = npg.params().cpu().double()
        tag = (cid, clamp, step)
        e = rel_l2(got - theta.double(), new_ref - theta.double())
        assert e < budget, (tag, e)
        for k in ("alpha", "kl_dist", "surr_after", "surr_before"):
            assert abs(out[k] - ref[k]) <= budget * max(abs(ref[k]), 1e-6 if k != "surr_before" else 1e-3), (tag, k, out[k], ref[k])
        assert (got[ls0:] >= MIN_LOG_STD).all(), tag
        ref_theta = new_ref
    if clamp:
        assert (new_ref[ls0:] == MIN_LOG_STD).any() and (got[ls0:] == MIN_LOG_STD).any(), "the clamp did not bind"
    # the policy the handle now runs is the one npg_params() describes
    theta_new = npg.params().cpu()
    ws, bs, ls = pol.unflatten(theta_new.double())
    fresh = engine()
    kw = c["kw"]
    fresh.load_policy([w.float() for w in ws], [b.float() for b in bs], kw["nonlinearity"], kw.get("in_shift"),
                      kw.get("in_scale"), kw.get("out_shift"), kw.get("out_scale"), ls.float())
    ob = c["obs"][-(2 * c["q"]["R"] + 3):].cuda()
    _, mean = eng.policy_act(ob)
    _, mean_ref = fresh.policy_act(ob)
    assert torch.equal(mean, mean_ref), cid
    assert rel_to_max(mean.cpu(), pol.mean(theta_new.double(), ob.cpu())) <= REL["mean"], cid
    ones = torch.ones(ob.shape[0], pol.sizes[-1], device="cuda")
    assert torch.allclose(eng.policy_act(ob, ones)[0], fresh.policy_act(ob, ones)[0], rtol=2e-7, atol=0)


# ---------------------------------------------------------------------------------------------------
# GPU: what the library accepts and refuses, and guard zones at every shape


@pytest.mark.gpu
@pytest.mark.parametrize("cid", IDS + [c["id"] for c in REFUSED])
def test_library_accepts_and_refuses_as_restated(cid):
    """npg_init accepts every table case (with the restated parameter count) and refuses the REFUSED rows for the
    restated reason; after a refusal the handle's policy still runs policy_act."""
    from amp_extensions_b200 import _lib
    c = case_data(cid)
    q = npg_geometry(c["sizes"])
    assert q["ok"]
    eng = engine()
    load(eng, c)
    if q["refused"] is None:
        assert eng.npg_init(MIN_LOG_STD) == q["n_params"] == c["pol"].n_params
        return
    msg = {"blocks": "gradient accumulator", "smem": "do not fit in shared memory"}[q["refused"]]
    with pytest.raises(_lib.SimstepError, match=msg):
        eng.npg_init(MIN_LOG_STD)
    obs = c["obs"][:257]
    _, mean = eng.policy_act(obs.cuda())
    assert rel_to_max(mean.cpu(), c["pol"].mean(c["theta"].double(), obs)) <= REL["mean"], cid


GUARD_SCRIPT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "write_policy_guards.py")


def npg_buffers(c):
    """Guarded NPG buffers: theta, old_theta, old_pack, old_std, vpack, g, x, r, p, scalars, skip, partial, dst,
    pack_of, and the activation cache when the policy has a hidden layer."""
    return 14 + (npg_geometry(c["sizes"])["cache_w"] > 0)


@pytest.mark.gpu
def test_guard_zones_around_npg_buffers(tmp_path):
    out = str(tmp_path / "guards.npz")
    env = dict(os.environ, SIMSTEP_DEBUG_GUARDS="1")
    res = subprocess.run([sys.executable, GUARD_SCRIPT, out], env=env, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-3000:]
    z = np.load(out)
    for c in CASES:
        n0, n1, bad = z[c["id"]]
        assert n1 - n0 == npg_buffers(c) and bad == 0, (c["id"], n0, n1, bad)


# ---------------------------------------------------------------------------------------------------
# CPU: the restatement and the case table


def test_case_table_reaches_every_npg_branch():
    reached = set()
    for c in CASES + REFUSED:
        reached |= npg_branches(c)
    required = {("R", 64), ("R", 32), ("refused", "blocks"), ("refused", "smem"),
                ("refused by the block count alone",), ("refused by shared memory alone",),
                ("blocks", "kNpgMaxBlocks"), ("blocks", "kNpgMaxBlocks + 1"),
                ("cache", "none"), ("cache", "hidden activations"),
                ("act_dim > 32", True), ("act_dim > 32", False), ("policy lane passes", 1), ("policy lane passes", 2),
                ("policy lane passes", 4), ("policy buffers", "obs_dim wide"), ("policy buffers", "128 wide"),
                ("obs_dim", "kPolicyMaxIn"), ("a width of 1",), ("activation", "relu"), ("activation", "tanh"),
                ("transforms", "with a zero in_scale column"), ("rows", "one"), ("rows", "ragged last tile"),
                ("grid", "fewer tiles than SMs"), ("grid", "several tiles per CTA")}
    required |= {("items per thread", k) for k in (1, 2, 3)} | {("layers", L) for L in (1, 2, 3, 4)}
    required |= {("in mod 4", k) for k in range(4)} | {("out mod 4", k) for k in range(4)}
    required |= {("mask", m) for m in MASKS}
    for b in sorted(reached, key=str):
        print("reached:", *b)
    missing = required - reached
    assert not missing, f"branches no case reaches: {sorted(missing, key=str)}"
    for c in CASES + REFUSED:
        assert c["covers"] and policy_geometry(c["sizes"])["ok"], c["id"]


def test_restatement_places_the_known_shapes():
    """The placements the case table was built from."""
    q = {cid: npg_geometry(CASE[cid]["sizes"]) for cid in CASE}
    assert (q["polA"]["R"], q["polA"]["blocks"], q["polA"]["items"]) == (64, 591, 2)
    assert q["relu64"]["R"] == 32 and npg_geometry([40, 64, 48, 33, 12])["R"] == 32
    assert (q["blocks1536"]["blocks"], q["blocks1536"]["R"], q["blocks1536"]["refused"]) == (1536, 32, None)
    assert q["blocks1537"]["blocks"] == 1537 and q["blocks1537"]["refused"] == "blocks"
    assert npg_smem(CASE["blocks1537"]["sizes"], 32) <= SMEM_LIMIT
    assert q["smem_only"]["blocks"] == 1297 and q["smem_only"]["refused"] == "smem"
    assert (q["obs512"]["R"], q["obs512"]["items"]) == (32, 3)
    assert q["four_layer"]["R"] == 64 and len(q["four_layer"]["outs"]) == 4
    assert q["linear"]["cache_w"] == 0
    for cid in IDS:
        assert q[cid]["n_params"] == no.Policy(CASE[cid]["sizes"]).n_params


def test_masked_row_fills_and_selection():
    """poison fills exactly the masked rows with non-finite values; relu rows clear the margin; advantages are exact in
    fp32 partial sums."""
    valid = torch.tensor([1, 0, 0, 1, 0], dtype=torch.uint8)
    x = poison(torch.ones(5, 2), valid)
    assert torch.equal(x[valid.bool()], torch.ones(2, 2))
    assert torch.isnan(x[1]).all() and (x[2] == float("inf")).all() and (x[4] == float("nan")).sum() == 0
    for cid in ("relu64", "relu_tf", "width1"):
        c = case_data(cid)
        if c["act"] == "relu":
            for p in hidden_pre(c["pol"], c["theta"].double(), c["obs"]):
                assert (p.abs() > MASK_MARGIN * float(p.abs().max())).all()
        a = c["adv"]
        assert torch.equal(a * 64, (a * 64).round()) and float(a.abs().max()) <= 4
        assert float(a.sum()) == float(a.double().sum())
    tf = case_data("relu_tf")["kw"]
    assert float(tf["in_scale"][ZERO_SCALE_COL]) == 0.0
