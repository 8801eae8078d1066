"""The ensemble training step (simstep_train_grads / _train_step, csrc/train.cuh, csrc/train_api.inc) at every shape,
member count, batch size and optimiser state its launch code dispatches on, against three oracles.

1. The reference oracle: DynamicsModel.train_step's arithmetic (oracle/milo_oracle.py TrainOracle) in float64 on the
   fp32 parameters: loss, every weight and bias gradient.  Budgets of tests/test_train_gpu.py: loss 1e-3, gradients
   4e-3 of the tensor's largest entry; relu hidden layers under that file's sparse bounds.
2. The operand-rounded oracle: the same float64 evaluation on exactly the values the kernels consume - the prepared x
   ((v - mean) / scale in fp32, then cvt.rna.tf32), every stored activation (bias + accumulator in fp32, activation,
   cvt.rna.tf32), the final dY (round_rna(fp32(2 / (B S)) * e)), the hidden dY (round_rna(dH * mask), the mask from the
   rounded h) and the raw fp32 master weights as the tensor core reads them (WEIGHT_OPERAND, pinned by
   test_tensor_core_truncates_raw_fp32_weights).  What is left is the fp32 accumulation and, now and then, one tf32 ulp
   of an activation, so its bound (REL_ROUNDED) is far below the reference budget.  A relu unit whose pre-activation
   sits within the accumulation error of zero would flip its mask and break a per-entry bound, so relu batches are
   drawn from rows whose every hidden pre-activation clears MASK_MARGIN (select_rows) instead of loosening the bound.
3. The optimiser restatement: train_optim_batch_kernel in numpy float32, fmaf order included, from the exported
   parameters, gradients and first moments; within an ulp or so of the kernel's parameters and moments.

The CPU section restates the launch code's dispatch predicates and checks that the tables reach every branch, and
checks oracles 2 and 3 against oracle 1 and torch.optim.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import milo_oracle as mo
from tests import helpers as H

LOSS_REL = 1e-3
GRAD_REL = 4e-3
FROB_REL = 2.5e-2      # relu hidden layers against oracle 1: Frobenius norm (test_train_gpu.py)
# bound of the operand-rounded oracle, per tensor, relative to the tensor's largest entry (loss: relative).  Worst
# error measured on one B200 (1000 W power limit) over every case and batch of test_gradients_match_oracles, bound about
# twice that: loss 1.19e-5 (no_transform), weight gradients 8.70e-4 (plain_mixed), bias gradients 7.93e-4 (north_star).
# The gradients' worst is one tf32 ulp (2^-11 .. 2^-10 of the entry) of a dY entry that the fp32 accumulation puts on
# the other side of a rounding tie than the float64 one, seen undiluted where few rows are summed: both worsts are at
# B = 1, and at B >= 200 no gradient passes 3.2e-4.  The loss sees only fp32 accumulation.  cvt.rz instead of cvt.rna in the prep kernel moves the loss by up to 9e-4 and flips relu masks.
REL_ROUNDED = {"loss": 2.5e-5, "weight": 1.7e-3, "bias": 1.6e-3}
# relu rows are kept when every hidden pre-activation of oracle 2 lies further than this share of the layer's
# largest |pre-activation| from zero, with the sign oracle 1 gives it.  Kernel and oracle 2 evaluate the same operands,
# so their pre-activations differ by the fp32 accumulation (~1e-6 relative) plus, where an upstream activation rounds
# to the neighbouring tf32 value, about |w| * 2^-11 * |h| (~1e-5 relative): 1e-4 clears both by ten.
MASK_MARGIN = 1e-4

# id, S, A, N, hidden, dense, act, transform, the branch the row exists for
CASES = [
    dict(id="n1", S=226, A=28, N=1, hidden=[256, 256], dense=True, act="relu", transform=True,
         covers="N = 1, humanoid dims"),
    dict(id="n2_plain_tanh_pad", S=226, A=28, N=2, hidden=[300, 300], dense=False, act="tanh", transform=True,
         covers="o_pad 512, plain BW descriptors, non-dense feat0_of"),
    dict(id="plain_mixed", S=40, A=12, N=3, hidden=[96, 300, 64], dense=False, act="relu", transform=True,
         covers="widths differing layer to layer in a plain net: kdg and k_pad differ per layer"),
    dict(id="n5_wide", S=64, A=8, N=5, hidden=[128] * 3, dense=True, act="relu", transform=True,
         covers="first layer in the wide epilogue (kb_x + kb_h <= 4), later layers narrow"),
    dict(id="n6_dense_tanh", S=46, A=10, N=6, hidden=[200, 200], dense=True, act="tanh", transform=True,
         covers="N = 6, tanh through dense connections (dgrad K spans two layers' dY)"),
    dict(id="n7_odd", S=45, A=7, N=7, hidden=[64, 64], dense=True, act="relu", transform=True,
         covers="odd S and A, N = 7, XP = 64: ragged wgrad n-tiles"),
    dict(id="n8", S=256, A=16, N=8, hidden=[256, 256], dense=True, act="relu", transform=True,
         covers="N = 8, S = 256"),
    dict(id="linear", S=30, A=6, N=3, hidden=[], dense=True, act="relu", transform=True,
         covers="L = 0: no dgrad, map_h aliases map_x, dh pitch 32"),
    dict(id="deep_dense", S=24, A=4, N=2, hidden=[64] * 8, dense=True, act="relu", transform=True,
         covers="36 BW transposes, 2L + 4 partial regions"),
    dict(id="deep_plain_tanh", S=24, A=4, N=2, hidden=[64] * 8, dense=False, act="tanh", transform=True,
         covers="eight chained plain dgrads"),
    dict(id="ragged_widths", S=226, A=28, N=2, hidden=[1, 65, 257], dense=True, act="relu", transform=True,
         covers="width 1 (255 padded units), 257 (o_pad 512)"),
    dict(id="s257", S=257, A=8, N=2, hidden=[64], dense=True, act="relu", transform=True,
         covers="SP = 512: two-tile final layer, two wgrad m-tiles, loss width 512"),
    dict(id="no_transform", S=226, A=28, N=4, hidden=[512, 512], dense=True, act="relu", transform=False,
         covers="prep and loss without transforms"),
    dict(id="a0", S=32, A=0, N=2, hidden=[64], dense=True, act="relu", transform=True,
         covers="null action pointer"),
    dict(id="north_star", S=226, A=28, N=4, hidden=[512] * 4, dense=True, act="relu", transform=True,
         covers="the shape that is trained in practice"),
]
CASE = {c["id"]: c for c in CASES}
IDS = [c["id"] for c in CASES]
MAX_ROWS = 1029
# one handle sized MAX_ROWS runs these in order (large -> small -> large: rows of an earlier, larger batch are left
# in the padded workspace); B = 256 also runs on a handle sized exactly 256 (B == Bp)
BATCH_ORDER = [1029, 200, 1, 256, 257]
EXACT = 256
POOL = 8192
OPTIM_CASES = ["linear", "plain_mixed", "deep_dense", "s257", "north_star"]
OPTIMS = {"sgd": dict(optim="sgd", lr=0.05, momentum=0.9, beta2=0.999, eps=1e-8, steps=3),
          "adam": dict(optim="adam", lr=1e-3, momentum=0.9, beta2=0.99, eps=1e-6, steps=12)}
CLIPS = ["off", "mixed", "loose"]     # grad_clip 0; the median member norm (binds for some members); 1e6 (binds for none)
OPTIM_B = 200


# ---------------------------------------------------------------------------------------------------
# operand formats and the oracles (CPU)


def rna(t):
    """fp32 -> tf32 round to nearest, ties away from zero (cvt.rna.tf32.f32), as fp32."""
    b = t.detach().float().contiguous().view(torch.int32)
    return ((b + 0x1000) & ~0x1FFF).view(torch.float32)


def trunc(t):
    """fp32 -> tf32 by dropping the 13 low mantissa bits."""
    b = t.detach().float().contiguous().view(torch.int32)
    return (b & ~0x1FFF).view(torch.float32)


# what the tensor core reads of a raw fp32 master weight (test_tensor_core_truncates_raw_fp32_weights)
WEIGHT_OPERAND = trunc

_cache = {}


def case_data(cid):
    """Parameters, transforms, the row pool and each member's batch rows of a case (seeded, cached)."""
    if cid in _cache:
        return _cache[cid]
    c = dict(CASE[cid])
    seed = 200 + IDS.index(cid)
    c["ws"], c["bs"] = mo.init_ensemble(c["S"], c["A"], c["hidden"], c["N"], dense_connect=c["dense"], base_seed=seed)
    c["pool"] = H.synth_dataset(POOL, c["S"], c["A"], seed)
    c["tf"] = mo.get_transformations(*c["pool"]) if c["transform"] else None
    c["rows"] = [select_rows(c, k, seed) for k in range(c["N"])]
    _cache[cid] = c
    return c


def batch(c, B):
    """[N, B, dim] state, action, next state: member k's first B selected rows."""
    return tuple(torch.stack([t[c["rows"][k][:B]] for k in range(c["N"])]).contiguous() for t in c["pool"])


def forward(c, k, s, a, rounded):
    """(inputs of every layer, hidden activations, hidden pre-activations, prediction, weights) of member k in float64,
    on the reference's values (oracle 1) or on the operands the kernels consume (oracle 2)."""
    if c["transform"]:
        ms, ss, ma, sa = c["tf"][:4]
        if rounded:   # train_prep_kernel: (v - mean) / scale in fp32 (a true division), then round
            x = rna(torch.cat([(s.float() - ms) / ss, (a.float() - ma) / sa], dim=1)).double()
        else:
            x = torch.cat([(s.double() - ms.double()) / ss.double(), (a.double() - ma.double()) / sa.double()], dim=1)
    else:
        x = torch.cat([s, a], dim=1)
        x = rna(x).double() if rounded else x.double()
    ws = [WEIGHT_OPERAND(w).double() if rounded else w.double() for w in c["ws"][k]]
    bs = [b.double() for b in c["bs"][k]]
    act = torch.relu if c["act"] == "relu" else torch.tanh
    inps, hs, pres = [x], [], []
    for w, b in zip(ws[:-1], bs[:-1]):
        pre = torch.nn.functional.linear(inps[-1], w, b)
        h = rna(act(pre.float())).double() if rounded else act(pre)
        pres.append(pre)
        hs.append(h)
        inps.append(torch.cat([inps[-1], h], dim=1) if c["dense"] else h)
    return inps, hs, pres, torch.nn.functional.linear(inps[-1], ws[-1], bs[-1]), ws


def oracle_grads(c, k, s, a, s2, rounded):
    """Oracle 1 (rounded False) or 2: (loss, [weight gradient per layer], [bias gradient per layer]) of member k."""
    B, S, L = s.shape[0], c["S"], len(c["hidden"])
    inps, hs, _, pred, ws = forward(c, k, s, a, rounded)
    if rounded:
        t = s2.float() - s.float()
        if c["transform"]:
            t = (t - c["tf"][4]) / c["tf"][5]
        e = pred - t.double()
        gscale = torch.tensor(2.0, dtype=torch.float32) / (torch.tensor(float(B)) * torch.tensor(float(S)))
        dy = rna(e.float() * gscale).double()
    else:
        t = s2.double() - s.double()
        if c["transform"]:
            t = (t - c["tf"][4].double()) / c["tf"][5].double()
        e = pred - t
        dy = e * (2.0 / (B * S))
    loss = float((e * e).mean())
    dys = [None] * L + [dy]
    X = c["S"] + c["A"]
    for j in range(L - 1, -1, -1):
        # dH_j: every layer that reads h_j (all later ones with dense connections, else the next), one K-concat
        readers = range(j + 1, L + 1) if c["dense"] else [j + 1]
        off = X + sum(c["hidden"][:j]) if c["dense"] else 0
        dh = torch.cat([dys[l] for l in readers], dim=1) @ torch.cat(
            [ws[l][:, off:off + c["hidden"][j]] for l in readers], dim=0)
        if rounded:   # train_mask_kernel: mask from the stored (rounded) h, product in fp32, then round
            h = hs[j].float()
            m = (h > 0).float() if c["act"] == "relu" else 1.0 - h * h
            dys[j] = rna(dh.float() * m).double()
        else:
            h = hs[j]
            m = (h > 0).double() if c["act"] == "relu" else 1.0 - h * h
            dys[j] = dh * m
    gw = [dys[l].t() @ inps[l] for l in range(L + 1)]
    gb = [dys[l].sum(0) for l in range(L + 1)]
    return loss, gw, gb


def select_rows(c, k, seed):
    """MAX_ROWS pool rows for member k (its own permutation).  relu: only rows whose every hidden pre-activation of
    oracle 2 clears MASK_MARGIN of the layer's scale with the sign oracle 1 gives it."""
    g = torch.Generator().manual_seed(1000 * seed + k)
    perm = torch.randperm(POOL, generator=g)
    if c["act"] != "relu" or not c["hidden"]:
        return perm[:MAX_ROWS]
    s, a, _ = c["pool"]
    keep, scale = [], None
    for chunk in perm.split(1024):
        p1 = forward(c, k, s[chunk], a[chunk], False)[2]
        p2 = forward(c, k, s[chunk], a[chunk], True)[2]
        if scale is None:
            scale = [float(p.abs().max()) for p in p2]
        ok = torch.ones(len(chunk), dtype=torch.bool)
        for q1, q2, sc in zip(p1, p2, scale):
            ok &= ((q2.abs() > MASK_MARGIN * sc) & ((q1 > 0) == (q2 > 0))).all(dim=1)
        keep.append(chunk[ok])
        if sum(len(x) for x in keep) >= MAX_ROWS:
            break
    rows = torch.cat(keep)
    assert len(rows) >= MAX_ROWS, (c["id"], k, len(rows))
    return rows[:MAX_ROWS]


def rel_to_max(x, ref):
    x, ref = np.asarray(x, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    return float(np.abs(x - ref).max() / max(np.abs(ref).max(), 1e-30))


def check_sparse(x, ref, what):
    """test_train_gpu.py's bound for relu hidden layers against the fp32 reference: Frobenius, median, percentiles."""
    x, ref = np.asarray(x, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    d = np.abs(x - ref) / max(np.abs(ref).max(), 1e-30)
    assert np.linalg.norm(x - ref) <= FROB_REL * np.linalg.norm(ref), what
    assert np.median(d) <= GRAD_REL, what
    if x.ndim == 2:
        assert (d <= GRAD_REL).mean() >= 0.95, what
        assert (d <= 10 * GRAD_REL).mean() >= 0.997, what


# ---------------------------------------------------------------------------------------------------
# oracle 3: train_optim_batch_kernel in float32

f32 = np.float32


def fmaf(a, b, c):
    """float32 fmaf: the product of two floats is exact in float64; one rounding of the sum (a double rounding can
    differ from the fused result by an ulp in rare ties)."""
    return (np.asarray(a, np.float64) * np.asarray(b, np.float64) + np.asarray(c, np.float64)).astype(f32)


def clip_coef(clip, sumsq):
    """min(1, clip / (fp32(sqrt(sumsq)) + 1e-6)), sumsq the member's float64 sum of squared gradients."""
    if clip <= 0:
        return f32(1)
    c = f32(clip) / (f32(np.sqrt(sumsq)) + f32(1e-6))
    return min(c, f32(1))


def optim_step(o, step, clip, p, g, m, v):
    """One member's update: flat float32 parameters, gradients, first and second moments -> (p, m, v) after it.
    step counts from 1 at the first step after train_init."""
    lr, mom, b2, eps = f32(o["lr"]), f32(o["momentum"]), f32(o["beta2"]), f32(o["eps"])
    grad = g * clip_coef(clip, float(np.sum(g.astype(np.float64) ** 2)))
    if o["optim"] == "sgd":
        buf = grad if step == 1 else fmaf(mom, m, grad)
        return fmaf(-lr, fmaf(mom, buf, grad), p), buf, v          # w -= lr * x contracts to one fma
    bc1 = f32(1.0 - float(mom) ** step)
    bc2 = f32(1.0 - float(b2) ** step)
    m1 = fmaf(mom, m, (f32(1) - mom) * grad)
    v1 = fmaf(b2, v, (f32(1) - b2) * grad * grad)
    denom = np.sqrt(v1) / np.sqrt(bc2) + eps
    return fmaf(-(lr / bc1), m1 / denom, p), m1, v1


def flat(ws, bs, k):
    return np.concatenate([t.numpy().ravel() for pair in zip(ws[k], bs[k]) for t in pair])


# ---------------------------------------------------------------------------------------------------
# GPU: engines


def train_engine(c, max_rows, optim="sgd"):
    from amp_extensions_b200.engine import Engine
    eng = Engine(c["S"], c["A"], c["N"], c["hidden"], dense_connect=c["dense"], activation=c["act"],
                 transform=c["transform"], precision="tf32")
    o = OPTIMS[optim]
    eng.train_init(max_rows, optim=o["optim"], lr=o["lr"], momentum=o["momentum"], beta2=o["beta2"], eps=o["eps"])
    eng.load_ensemble(c["ws"], c["bs"], c["tf"])
    return eng


def cuda(*ts):
    return tuple(t.cuda() for t in ts)


# ---------------------------------------------------------------------------------------------------
# GPU: loss and gradients against oracles 1 and 2


@pytest.mark.gpu
@pytest.mark.parametrize("cid", IDS)
def test_gradients_match_oracles(cid):
    c = case_data(cid)
    L = len(c["hidden"])
    big = train_engine(c, MAX_ROWS)
    runs = [(big, B) for B in BATCH_ORDER] + [(train_engine(c, EXACT), EXACT)]
    worst = {}
    for eng, B in runs:
        s, a, s2 = batch(c, B)
        loss = eng.train_grads(*cuda(s, a, s2)).cpu().numpy()
        gw, gb = eng.train_export(eng.TRAIN_GRADS)
        for k in range(c["N"]):
            l1, gw1, gb1 = oracle_grads(c, k, s[k], a[k], s2[k], False)
            l2, gw2, gb2 = oracle_grads(c, k, s[k], a[k], s2[k], True)
            tag = (cid, B, k)
            assert abs(loss[k] - l1) <= LOSS_REL * l1, (tag, loss[k], l1)
            e = abs(loss[k] - l2) / l2
            worst[B, "loss"] = max(worst.get((B, "loss"), 0.0), e)
            assert e <= REL_ROUNDED["loss"], (tag, "loss (operand-rounded oracle)", e)
            for l in range(L + 1):
                for what, x, r1, r2 in (("weight", gw[k][l], gw1[l], gw2[l]), ("bias", gb[k][l], gb1[l], gb2[l])):
                    if c["act"] == "relu" and l < L:
                        check_sparse(x, r1, (tag, l, what))
                    else:
                        assert rel_to_max(x, r1) <= GRAD_REL, (tag, l, what, rel_to_max(x, r1))
                    e = rel_to_max(x, r2)
                    worst[B, what] = max(worst.get((B, what), 0.0), e)
                    assert e <= REL_ROUNDED[what], (tag, l, what, "operand-rounded oracle", e)
    print(f"worst against the operand-rounded oracle: {cid}", {k: f"{v:.2e}" for k, v in worst.items()})


# ---------------------------------------------------------------------------------------------------
# GPU: the optimiser against its float32 restatement


def optim_runs(c, eng, optim, clip_mode, rows0):
    """train_init(optim) on `eng` (parameters stay: a re-init restarts the step count and the moments), then the
    optimiser's steps, each checked against optim_step.  Returns the clip coefficients of the first step."""
    o = OPTIMS[optim]
    eng.train_init(OPTIM_B, optim=o["optim"], lr=o["lr"], momentum=o["momentum"], beta2=o["beta2"], eps=o["eps"])
    N = c["N"]
    v = None
    clip, coefs = 0.0, None
    s_all, a_all, s2_all = c["pool"]
    for step in range(1, o["steps"] + 1):
        idx = torch.stack([c["rows"][k].roll(-(rows0 + 37 * step))[:OPTIM_B] for k in range(N)])
        s, a, s2 = cuda(s_all[idx], a_all[idx], s2_all[idx])
        pw, pb = eng.train_export(eng.TRAIN_PARAMS)
        mw, mb = eng.train_export(eng.TRAIN_MOMENTS)
        eng.train_grads(s, a, s2)
        g1 = eng.train_export(eng.TRAIN_GRADS)
        if step == 1:
            norms = np.array([np.sqrt(np.sum(flat(*g1, k).astype(np.float64) ** 2)) for k in range(N)])
            clip = {"off": 0.0, "mixed": float(np.median(norms)), "loose": 1e6}[clip_mode]
            coefs = [clip_coef(clip, n * n) for n in norms]
            v = [np.zeros_like(flat(pw, pb, k)) for k in range(N)]
        eng.train_step(s, a, s2, grad_clip=clip)
        g2 = eng.train_export(eng.TRAIN_GRADS)
        nw, nb = eng.train_export(eng.TRAIN_PARAMS)
        n_mw, n_mb = eng.train_export(eng.TRAIN_MOMENTS)
        for k in range(N):
            g = flat(*g2, k)
            assert np.array_equal(flat(*g1, k), g), "train_step's gradients differ from train_grads' on the same batch"
            p0 = flat(pw, pb, k)
            p, m, v[k] = optim_step(o, step, clip, p0, g, flat(mw, mb, k), v[k])
            got_p, got_m = flat(nw, nb, k), flat(n_mw, n_mb, k)
            tag = (c["id"], optim, clip_mode, step, k)
            assert np.abs(got_p - p0).max() > 0, tag
            # one ulp of the result (a double-rounded fmaf), a few of the step itself
            tol = np.spacing(np.abs(p)) + 4 * np.spacing(np.abs(p - p0))
            assert (np.abs(got_p - p) <= tol).all(), (tag, "parameters", float(np.abs(got_p - p).max()))
            assert (np.abs(got_m - m) <= 2 * np.spacing(np.abs(m))).all(), (tag, "moment", float(np.abs(got_m - m).max()))
    return coefs


@pytest.mark.gpu
@pytest.mark.parametrize("cid", OPTIM_CASES)
def test_optimiser_matches_restatement(cid):
    c = case_data(cid)
    eng = train_engine(c, OPTIM_B)
    for i, (optim, clip_mode) in enumerate((o, m) for o in OPTIMS for m in CLIPS):
        coefs = optim_runs(c, eng, optim, clip_mode, 100 * i)
        if clip_mode == "mixed":
            assert min(coefs) < 1 and max(coefs) == 1, coefs     # binds for some members and not for the others
        else:
            assert all(x == 1 for x in coefs), coefs


# ---------------------------------------------------------------------------------------------------
# GPU: what the tensor core reads of a weight, and the trained handle's env step


@pytest.mark.gpu
def test_tensor_core_truncates_raw_fp32_weights():
    """A linear no-transform handle evaluated on one-hot rows with zero biases returns every weight as the tensor core
    consumed it (one product, fp32 accumulation, exact).  A training handle keeps raw fp32 weights: the tensor core
    reads their top 19 bits, truncation.  A tf32 handle without train_init holds the cvt.rna-packed weights."""
    from amp_extensions_b200.engine import Engine
    S, A, N = 30, 6, 2
    g = torch.Generator().manual_seed(3)
    ws = [[torch.randn(S, S + A, generator=g)] for _ in range(N)]
    low = torch.randint(0, 0x2000, (N, S, S + A), generator=g, dtype=torch.int32)
    low.view(-1)[:4] = torch.tensor([0x1000, 0x0FFF, 0x1FFF, 0x0001], dtype=torch.int32)   # ties and both sides
    for k in range(N):
        ws[k][0] = ((ws[k][0].view(torch.int32) & ~0x1FFF) | low[k]).view(torch.float32)
    bs = [[torch.zeros(S)] for _ in range(N)]
    eye = torch.eye(S + A)
    s, a = eye[:, :S].contiguous().cuda(), eye[:, S:].contiguous().cuda()
    outs = {}
    for train in (True, False):
        eng = Engine(S, A, N, [], transform=False, precision="tf32")
        if train:
            eng.train_init(16)
        eng.load_ensemble(ws, bs, None)
        outs[train] = eng.forward(s, a).cpu()          # [N, S + A, S]: out[k, i, o] = W_k[o, i]
        eng.close()
    for k in range(N):
        w = ws[k][0]
        assert not torch.equal(trunc(w), rna(w))
        assert torch.equal(outs[True][k].t(), trunc(w)), "training handle: the tensor core does not truncate"
        assert torch.equal(outs[False][k].t(), rna(w)), "inference handle: weights not cvt.rna-packed"


@pytest.mark.gpu
@pytest.mark.parametrize("cid", ["north_star", "n2_plain_tanh_pad", "linear"])
def test_trained_handle_env_step_matches_truncated_weights(cid):
    """After a few SGD steps, the handle's env forward against the step matrix's operand-rounded oracle on the
    exported raw weights, truncated as the tensor core reads them, at the tf32 bound of that oracle."""
    from tests import test_step_matrix_gpu as M
    c = case_data(cid)
    eng = train_engine(c, OPTIM_B)
    for step in range(4):
        s, a, s2 = batch(c, OPTIM_B)
        eng.train_step(*cuda(s, a, s2.roll(step, dims=1)), grad_clip=1.0)
    ws, bs = eng.train_export(eng.TRAIN_PARAMS)
    assert any(not torch.equal(ws[0][l], c["ws"][0][l]) for l in range(len(ws[0])))
    cc = dict(c, ws=[[trunc(w) for w in m] for m in ws], bs=bs)   # exact tf32 values: rna leaves them unchanged
    g = torch.Generator().manual_seed(11)
    E = 257
    s = c["pool"][0][torch.randint(0, POOL, (E,), generator=g)]
    a = c["pool"][1][torch.randint(0, POOL, (E,), generator=g)]
    fwd = eng.forward(s.cuda(), a.cuda())
    ref = M.rounded_deltas(cc, s, a, "tf32")
    M.assert_close(fwd, ref, float(ref.abs().max()), rel=M.REL_ROUNDED["tf32"], what=f"{cid} trained forward")


@pytest.mark.gpu
@pytest.mark.parametrize("cid", ["linear", "deep_plain_tanh"])
@pytest.mark.parametrize("B", [256, 200])
def test_graph_replay_equals_eager_steps(cid, B):
    c = case_data(cid)
    outs = []
    for use_graph in (False, True):
        eng = train_engine(c, B, optim="adam")
        for step in range(5):
            s, a, s2 = batch(c, B)
            fn = eng.train_step_graph if use_graph else eng.train_step
            loss = fn(*cuda(s, a, s2.roll(step, dims=1)), grad_clip=0.3).clone()
        outs.append((loss.cpu(),) + eng.train_export(eng.TRAIN_PARAMS) + eng.train_export(eng.TRAIN_MOMENTS))
        assert eng.check_guards() == (0, 0)      # no guard zones without SIMSTEP_DEBUG_GUARDS=1
    assert torch.equal(outs[0][0], outs[1][0])
    for k in range(c["N"]):
        assert np.array_equal(flat(outs[0][1], outs[0][2], k), flat(outs[1][1], outs[1][2], k))
        assert np.array_equal(flat(outs[0][3], outs[0][4], k), flat(outs[1][3], outs[1][4], k))


# ---------------------------------------------------------------------------------------------------
# GPU: guard zones around every training buffer (SIMSTEP_DEBUG_GUARDS is read when a handle is created)

GUARD_SCRIPT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "write_train_guards.py")


def train_buffers(c):
    """Guarded training buffers: x, hb, pred, xt, dy, dyt, dh, gb, mb, vb, partial, loss, sumsq; g, m, v per layer;
    bw per hidden layer."""
    L = len(c["hidden"])
    return 13 + 3 * (L + 1) + L


@pytest.mark.gpu
def test_guard_zones_around_training_buffers(tmp_path):
    out = str(tmp_path / "guards.npz")
    env = dict(os.environ, SIMSTEP_DEBUG_GUARDS="1")
    res = subprocess.run([sys.executable, GUARD_SCRIPT, out], env=env, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-3000:]
    z = np.load(out)
    for c in CASES:
        for handle in ("max", "exact"):
            n, bad = z[f"{c['id']}_{handle}"]
            assert n == train_buffers(c) and bad == 0, (c["id"], handle, n, bad)


# ---------------------------------------------------------------------------------------------------
# CPU: the dispatch predicates of csrc/train_api.inc and api.cu, and the oracles themselves

K_BLOCK_N, ROW_TILE, BK = 256, 256, 32        # kBlockN, row_align = 2 * kBlockM, tf32 elements per swizzle row
WIDE_STAGES = 4                               # GemmPlan<2, true>::kStages


def rup(x, m):
    return (x + m - 1) // m * m


def geometry(c):
    """simstep_create's layer table for a tf32 handle: per layer (o_pad, k_pad, kb_x, kb_h), and SP."""
    S, A, L, hid, dense = c["S"], c["A"], len(c["hidden"]), c["hidden"], c["dense"]
    XP = rup(S + A, 64)
    hp = [rup(h, K_BLOCK_N) for h in hid]
    hcol = [sum(hp[:i]) for i in range(L)]
    layers = []
    for l in range(L + 1):
        o_pad = hp[l] if l < L else rup(S, K_BLOCK_N)
        if dense or l == 0:
            kb_h = (hcol[l - 1] + hp[l - 1]) // BK if dense and l > 0 else 0
            layers.append(dict(o_pad=o_pad, kb_x=XP // BK, kb_h=kb_h, k_pad=XP + kb_h * BK))
        else:
            layers.append(dict(o_pad=o_pad, kb_x=0, kb_h=hp[l - 1] // BK, k_pad=hp[l - 1]))
    return dict(XP=XP, SP=rup(S, K_BLOCK_N), layers=layers)


def train_branches(c, B, B_cap):
    """The launch paths one train_grads / train_step of case c with B rows on a handle sized B_cap takes."""
    g, L, b = geometry(c), len(c["hidden"]), set()
    for ly in g["layers"][:L]:   # launch_gemm: two epilogue groups when the store mode's whole K fits the short ring
        b.add(("forward epilogue", "wide" if ly["kb_x"] + ly["kb_h"] <= WIDE_STAGES else "narrow"))
    if L == 0:
        b.add(("L == 0: no dgrad, map_h = map_x",))
    else:   # train_build_descs: BW transposes
        b.add(("BW descriptors", "L(L+1)/2 dense" if c["dense"] else "L plain"))
        if not c["dense"]:
            b.add(("feat0_of / kdg", "non-dense"))
    b.add(("final layer n-tiles", g["SP"] // K_BLOCK_N))
    for ly in g["layers"]:
        b.add(("wgrad k_pad % 256", "zero" if ly["k_pad"] % K_BLOCK_N == 0 else "ragged"))
    Bp = rup(B_cap, ROW_TILE)
    b.add(("forward m-tiles", "1" if Bp == ROW_TILE else ">= 2"))
    b.add(("batch", "B < Bp" if B < Bp else "B == Bp"))
    if B < B_cap:
        b.add(("batch", "B < B_cap"))
    b.add(("activation", c["act"]))
    b.add(("transform", c["transform"]))
    if c["A"] == 0:
        b.add(("A == 0",))
    b.add(("N", c["N"]))
    return b


def n_bw(c):
    L = len(c["hidden"])
    return L * (L + 1) // 2 if c["dense"] else L


def test_case_table_reaches_every_train_branch():
    reached = set()
    for c in CASES:
        for B in BATCH_ORDER:
            reached |= train_branches(c, B, MAX_ROWS)
        reached |= train_branches(c, EXACT, EXACT)
    for cid in OPTIM_CASES:
        reached |= train_branches(CASE[cid], OPTIM_B, OPTIM_B)
        reached |= {("optimiser", o, m) for o in OPTIMS for m in CLIPS}
    required = {("forward epilogue", "wide"), ("forward epilogue", "narrow"), ("L == 0: no dgrad, map_h = map_x",),
                ("BW descriptors", "L(L+1)/2 dense"), ("BW descriptors", "L plain"), ("feat0_of / kdg", "non-dense"),
                ("final layer n-tiles", 1), ("final layer n-tiles", 2), ("wgrad k_pad % 256", "zero"),
                ("wgrad k_pad % 256", "ragged"), ("forward m-tiles", "1"), ("forward m-tiles", ">= 2"),
                ("batch", "B < Bp"), ("batch", "B == Bp"), ("batch", "B < B_cap"), ("activation", "relu"),
                ("activation", "tanh"), ("transform", True), ("transform", False), ("A == 0",)}
    required |= {("N", n) for n in range(1, 9)} | {("optimiser", o, m) for o in OPTIMS for m in CLIPS}
    for b in sorted(reached, key=str):
        print("reached:", *b)
    missing = required - reached
    assert not missing, f"branches no case reaches: {sorted(missing, key=str)}"
    assert n_bw(CASE["deep_dense"]) == 36 and 2 * len(CASE["deep_dense"]["hidden"]) + 4 == 20
    # plain_mixed: every layer reads a different K, every dgrad a different kdg
    lys = geometry(CASE["plain_mixed"])["layers"]
    assert len({ly["k_pad"] for ly in lys}) == 3 and len({ly["o_pad"] for ly in lys[1:]}) == 2
    assert [ly["o_pad"] for ly in geometry(CASE["ragged_widths"])["layers"][:3]] == [256, 256, 512]
    for c in CASES:
        assert c["covers"] and len(c["hidden"]) <= 8 and c["N"] <= 8


def test_operand_rounded_oracle_is_the_reference_oracle_without_rounding():
    """Oracle 2 is oracle 1's evaluation with the operand rounding switched on (so without it, it is oracle 1 bit for
    bit); oracle 1 is float64 autograd through TrainOracle's graph; the rounding moves the gradients by a tf32-sized
    amount."""
    for cid in ("n7_odd", "n2_plain_tanh_pad", "no_transform", "linear", "a0"):
        c = case_data(cid)
        s, a, s2 = (t[0] for t in batch(c, 64))
        l1, gw1, gb1 = oracle_grads(c, 0, s, a, s2, False)
        # the same oracle spelled as TrainOracle's autograd graph, in float64
        ws = [w.double().requires_grad_() for w in c["ws"][0]]
        bs = [b.double().requires_grad_() for b in c["bs"][0]]
        x = torch.cat([s.double(), a.double()], dim=1)
        t = s2.double() - s.double()
        if c["transform"]:
            tf = [v.double() for v in c["tf"]]
            x = torch.cat([(s.double() - tf[0]) / tf[1], (a.double() - tf[2]) / tf[3]], dim=1)
            t = (t - tf[4]) / tf[5]
        loss = torch.nn.functional.mse_loss(mo.mlp_forward(ws, bs, x, c["dense"], c["act"]), t)
        loss.backward()
        assert abs(l1 - loss.item()) <= 1e-12 * loss.item()
        for l in range(len(ws)):
            assert rel_to_max(gw1[l], ws[l].grad) < 1e-12 and rel_to_max(gb1[l], bs[l].grad) < 1e-12, (cid, l)
        l2, gw2, gb2 = oracle_grads(c, 0, s, a, s2, True)
        err = max(rel_to_max(x, r) for x, r in zip(gw2 + gb2, gw1 + gb1))
        assert 1e-5 < err < GRAD_REL, (cid, err)
        assert abs(l2 - l1) <= LOSS_REL * l1


def test_rna_and_trunc_round_as_the_hardware_formats():
    x = torch.tensor([1.0 + 2 ** -11, 1.0 + 2 ** -11 - 2 ** -23, -(1.0 + 2 ** -11), 1.0 + 3 * 2 ** -11,
                      1.0 + 2 ** -10 - 2 ** -23], dtype=torch.float32)
    assert rna(x).tolist() == [1.0 + 2 ** -10, 1.0, -(1.0 + 2 ** -10), 1.0 + 2 ** -9, 1.0 + 2 ** -10]
    assert trunc(x).tolist() == [1.0, 1.0, -1.0, 1.0 + 2 ** -10, 1.0]


@pytest.mark.parametrize("optim", list(OPTIMS))
def test_optimiser_restatement_matches_torch_optim(optim):
    """oracle 3 against torch.optim.SGD(nesterov=True) / torch.optim.Adam with clip_grad_norm_ on CPU fp32, three
    members, every clip mode, over the optimiser's steps and a restart."""
    o = OPTIMS[optim]
    g = torch.Generator().manual_seed(4)
    shapes = [(64, 40), (64,), (30, 104), (30,)]
    for clip_mode in CLIPS:
        for member in range(3):
            ps = [torch.randn(sh, generator=g) for sh in shapes]
            grads = [[torch.randn(sh, generator=g) * (0.5 + member) for sh in shapes] for _ in range(o["steps"])]
            clip = {"off": 0.0, "mixed": 100.0, "loose": 1e6}[clip_mode]   # norms ~40, 110, 190
            tp = [torch.nn.Parameter(p.clone()) for p in ps]
            if optim == "sgd":
                opt = torch.optim.SGD(tp, lr=o["lr"], momentum=o["momentum"], nesterov=True, foreach=False)
            else:
                opt = torch.optim.Adam(tp, lr=o["lr"], betas=(o["momentum"], o["beta2"]), eps=o["eps"], foreach=False)
            p = np.concatenate([x.numpy().ravel() for x in ps])
            m, v = np.zeros_like(p), np.zeros_like(p)
            for step, gs in enumerate(grads, 1):
                for t, gr in zip(tp, gs):
                    t.grad = gr.clone()
                if clip:
                    torch.nn.utils.clip_grad_norm_(tp, clip)
                opt.step()
                p0 = p
                p, m, v = optim_step(o, step, clip, p, np.concatenate([x.numpy().ravel() for x in gs]), m, v)
                want = np.concatenate([t.detach().numpy().ravel() for t in tp])
                moved = np.abs(want - p0).max()
                assert np.abs(p - want).max() <= 1e-5 * moved + 8 * np.spacing(np.abs(want).max()), \
                    (optim, clip_mode, member, step, float(np.abs(p - want).max()), float(moved))
