"""The env step (simstep_step / _step_cost / _discrepancy / _forward) at every shape, member count, precision, cost input
type and row alignment its launch code dispatches on, against two float64 oracles.

1. The reference oracle: the reference's arithmetic (dynamics.py:216-233, sim_env.py:140-173, linear_cost.py:111-152) in
   float64 on the fp32 weights, at test_parity_gpu.py's 1e-3 budget for tf32 and fp16 operands.
2. The operand-rounded oracle: the same float64 evaluation on exactly the values the kernels round - the packed weights,
   the prepared input rows and every hidden layer's stored activations, each rounded as csrc/ converts it (E::cvt and
   the hidden epilogue's pack32: tf32 round-to-nearest-away, fp16 round-to-nearest saturating at 65 504, bf16
   round-to-nearest) - for all three precisions.  What is left is the fp32 accumulation of the tensor cores, so its
   bound is far below 1e-3: a missing lo term, a wrong rounding mode or a bias read from a neighbouring padded tile
   shows up there long before it reaches the reference budget.

The CPU section restates the launch code's dispatch predicates and checks that the case table reaches every branch.
"""
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import milo_oracle as mo
from tests import helpers as H

REL = 1e-3
# bound of the operand-rounded oracle per precision (per element, relative to max(|ref|, scale)): what is left is the fp32
# accumulation and, where the fp32 and the float64 pre-activation of a hidden unit round to neighbouring operand values,
# one operand ulp of that activation.  Worst error measured on one B200 (1000 W) over every case and batch size of
# test_step_matches_oracles: tf32 1.54e-4, fp16 1.52e-4 (next state, no_transform), bf16 4.1e-4 (deltas, n8_s256); the
# discrepancy at most 7.0e-5
REL_ROUNDED = {"tf32": 3e-4, "fp16": 3e-4, "bf16": 1e-3}

# id, S, A, N, hidden, dense, act, transform, the branch the row exists for
CASES = [
    dict(id="n1", S=226, A=28, N=1, hidden=[256, 256], dense=True, act="relu", transform=True,
         covers="NM = 1 (discrepancy is 0), post_step_tma_kernel<.., 226>, humanoid termination"),
    dict(id="n2_plain_tanh_pad", S=226, A=28, N=2, hidden=[300, 300], dense=False, act="tanh", transform=True,
         covers="hidden widths padded to 512-column tiles, column-fused chain with tanh, no dense connections"),
    dict(id="n5_generic_tma", S=64, A=8, N=5, hidden=[128] * 3, dense=True, act="relu", transform=True,
         covers="NM = 5, post_step_tma_kernel<.., 0> with S = 0 mod 4"),
    dict(id="n6_s2mod4", S=46, A=10, N=6, hidden=[200, 200], dense=True, act="relu", transform=True,
         covers="NM = 6, S = 2 mod 4 row pairs in the generic TMA kernel"),
    dict(id="n7_odd", S=45, A=7, N=7, hidden=[64, 64], dense=True, act="relu", transform=True,
         covers="NM = 7, scalar post kernel, non-vector prep, unfused 'ss' pack with s' at round_up(S, 8)"),
    dict(id="n7_even", S=62, A=9, N=7, hidden=[96, 160], dense=True, act="relu", transform=True,
         covers="NM = 7 through the TMA and float2 post kernels, odd A with even S (non-vector prep, fused 'ss' rows)"),
    dict(id="n8_s256", S=256, A=16, N=8, hidden=[256, 256], dense=True, act="relu", transform=True,
         covers="S = kPostMaxElems, NM = 8, the largest TMA stage"),
    dict(id="linear", S=30, A=6, N=3, hidden=[], dense=True, act="relu", transform=True,
         covers="n_hidden = 0: the final layer alone, one launch per layer, never the chain"),
    dict(id="deep", S=24, A=4, N=2, hidden=[64] * 8, dense=True, act="relu", transform=True,
         covers="SIMSTEP_MAX_HIDDEN: a 9-layer chain"),
    dict(id="ragged_widths", S=226, A=28, N=2, hidden=[1, 65, 257], dense=True, act="relu", transform=True,
         covers="width 1, off-by-one tile and bk edges in the concat offsets"),
    dict(id="no_transform", S=226, A=28, N=4, hidden=[512, 512], dense=True, act="relu", transform=False,
         covers="prep without transforms, final epilogue without scale / shift"),
    dict(id="a0", S=32, A=0, N=2, hidden=[64], dense=True, act="relu", transform=True,
         covers="action_dim = 0: a null action pointer is accepted"),
    dict(id="xp_boundary", S=40, A=24, N=3, hidden=[128, 128], dense=True, act="tanh", transform=True,
         covers="S + A = 64 exactly (XP without padding)"),
    dict(id="square", S=16, A=16, N=3, hidden=[64, 64], dense=True, act="relu", transform=True,
         covers="S == A: 'sa' and 'ss' have the same width"),
]
CASE = {c["id"]: c for c in CASES}
IDS = [c["id"] for c in CASES]
BF16_CASES = ["n1", "n7_odd", "n8_s256", "square"]
STEP_PARAMS = [(i, p) for i in IDS for p in ("tf32", "fp16")] + [(i, "bf16") for i in BF16_CASES]
BATCHES = [1, 257, 1029]       # one row; one row past a 256-row tile; an odd count (trailing row of the row pairs)
CHUNK = 512                    # max_chunk_envs of the chunked run: 1029 rows are three chunks
COST_CASES = {"n7_odd": 100, "n6_s2mod4": 257, "n1": 257, "square": 100}   # case -> feature_dim D (neither a tile multiple)
INPUT_TYPES = ["s", "sa", "ss", "sas"]
HORIZON = 300


# ---------------------------------------------------------------------------------------------------
# case data and oracles (CPU)

_cache = {}


def case_data(cid):
    """Weights, transforms and per-batch inputs of a case (seeded, cached)."""
    if cid in _cache:
        return _cache[cid]
    c = dict(CASE[cid])
    seed = 100 + IDS.index(cid)
    c["ws"], c["bs"] = mo.init_ensemble(c["S"], c["A"], c["hidden"], c["N"], dense_connect=c["dense"], base_seed=seed)
    c["tf"] = mo.get_transformations(*H.synth_dataset(2048, c["S"], c["A"], seed))
    c["humanoid"] = c["S"] == 226
    _cache[cid] = c
    return c


def inputs(c, E, seed=0):
    g = torch.Generator().manual_seed(1000 * seed + E)
    s = H.humanoid_like_states(E, seed=E + seed) if c["humanoid"] else torch.randn(E, c["S"], generator=g)
    a = torch.randn(E, c["A"], generator=g)
    member = torch.randint(0, c["N"], (E,), generator=g, dtype=torch.int32)
    steps = torch.randint(0, HORIZON, (E,), generator=g, dtype=torch.int32)
    steps[: max(1, E // 8)] = HORIZON - 1      # done has both outcomes
    if E > 1:
        steps[-1] = 0
    return s, a, member, steps


def rounder(prec):
    """float64 copy of an fp32 tensor rounded to the operand format of `prec` (None: no rounding)."""
    from amp_extensions_b200.linear_cost import RBFLinearCost
    if prec is None:
        return lambda t: t.double()
    return lambda t: RBFLinearCost._round_operand(t, prec)


def reference_deltas(c, s, a):
    """Oracle 1: every member's un-normalised prediction [N, E, S], the reference's forward in float64."""
    x = torch.cat([s.double(), a.double()], dim=1)
    if c["transform"]:
        ms, ss, ma, sa = (t.double() for t in c["tf"][:4])
        x = torch.cat([(s.double() - ms) / ss, (a.double() - ma) / sa], dim=1)
    out = []
    for ws, bs in zip(c["ws"], c["bs"]):
        d = mo.mlp_forward([w.double() for w in ws], [b.double() for b in bs], x, c["dense"], c["act"])
        if c["transform"]:
            d = d * c["tf"][5].double() + c["tf"][4].double()
        out.append(d)
    return torch.stack(out)


def rounded_deltas(c, s, a, prec):
    """Oracle 2: oracle 1 evaluated on the values the kernels round, accumulated in float64.  prec None: no rounding,
    which must be oracle 1 bit for bit.  The prepared row is (x - mean) * (1 / scale) in fp32 (prep_input_kernel); a
    hidden activation is bias + accumulator in fp32, the activation, then the operand conversion (pack32)."""
    rnd = rounder(prec)
    if c["transform"]:
        ms, ss, ma, sa = c["tf"][:4]
        if prec is None:
            xs, xa = (s.double() - ms.double()) / ss.double(), (a.double() - ma.double()) / sa.double()
        else:
            xs, xa = (s.float() - ms) * (1.0 / ss), (a.float() - ma) * (1.0 / sa)
    else:
        xs, xa = s.float(), a.float()
    x = rnd(torch.cat([xs, xa], dim=1)) if prec is not None else torch.cat([xs.double(), xa.double()], dim=1)
    act64 = torch.relu if c["act"] == "relu" else torch.tanh
    out = []
    for ws, bs in zip(c["ws"], c["bs"]):
        inp = x
        for w, b in zip(ws[:-1], bs[:-1]):
            pre = torch.nn.functional.linear(inp, rnd(w), b.double())
            h = act64(pre) if prec is None else rnd(act64(pre.float()))
            inp = torch.cat([inp, h], dim=1) if c["dense"] else h
        d = torch.nn.functional.linear(inp, rnd(ws[-1]), bs[-1].double())
        if c["transform"]:
            d = d * c["tf"][5].double() + c["tf"][4].double()
        out.append(d)
    return torch.stack(out)


def oracle_step(c, s, a, member, steps, preds):
    """(next state f64, steps + 1, done, discrepancy) of the step on member deltas `preds`."""
    active = preds[member.long(), torch.arange(s.shape[0])]
    nxt = s.double() + active
    steps1 = steps.long() + 1
    done = steps1 >= HORIZON
    if c["humanoid"]:
        done = done | torch.from_numpy(mo.simenv_collided(nxt.numpy()) | mo.simenv_velocity_exploded(nxt.numpy()))
    return nxt, steps1, done, mo.discrepancy_from_preds(preds).double()


def scales(c, preds, disc_ref):
    """Per-output scales of assert_close: the state spread and the mean discrepancy (test_step_matches_oracle's), and
    the largest member delta of the batch - an element's operand error follows the magnitude of its whole row, and
    the states of the humanoid cases lie far outside the transforms' data."""
    s_next = c["tf"][1].mean().item() if c["transform"] else 1.0
    return s_next, max(disc_ref.mean().item(), 1e-30), float(preds.abs().max())


def rel_err(x, ref, scale):
    x, ref = x.detach().double().cpu(), ref.detach().double().cpu()
    return float(((x - ref).abs() / torch.maximum(ref.abs(), torch.full_like(ref, scale))).max()) if ref.numel() else 0.0


def assert_close(x, ref, scale, rel=REL, what=""):
    from tests.test_parity_gpu import assert_close as ac
    ac(x, ref, scale, rel=rel, what=what)


def threshold_margin(c, nxt_ref):
    """Distance of every row's tested quantities to their termination thresholds (inf without fall contacts)."""
    if not c["humanoid"]:
        return np.full(nxt_ref.shape[0], np.inf)
    from tests.test_parity_gpu import collision_margin
    ob = nxt_ref.numpy()
    return np.minimum(collision_margin(ob), np.abs(np.abs(ob[:, 136:]) - 100).min(1))


# ---------------------------------------------------------------------------------------------------
# GPU: engines

_engines = {}


def termination(c):
    """Humanoid fall contacts and velocity check at S = 226; elsewhere the handle's default, the horizon alone."""
    from amp_extensions_b200.engine import HumanoidTermination
    if c["humanoid"]:
        return HumanoidTermination(horizon=HORIZON, enable_velocity_check=True)
    return HumanoidTermination(horizon=HORIZON, fall_contact_bodies=())


def engine(cid, prec, chunk=0):
    key = (cid, prec, chunk)
    if key not in _engines:
        from amp_extensions_b200.engine import Engine
        c = case_data(cid)
        eng = Engine(c["S"], c["A"], c["N"], c["hidden"], dense_connect=c["dense"], activation=c["act"],
                     transform=c["transform"], precision=prec, max_chunk_envs=chunk)
        eng.load_ensemble(c["ws"], c["bs"], c["tf"] if c["transform"] else None)
        if c["humanoid"]:
            eng.set_termination(termination(c))
        _engines[key] = eng
    return _engines[key]


def cost_oracle(c, itype, D, seed=7):
    """RffCostOracle fitted on expert rows of input_type's width (and the host-side layer RBFLinearCost builds from the
    same seed)."""
    S, A = c["S"], c["A"]
    width = {"s": S, "sa": S + A, "ss": 2 * S, "sas": 2 * S + A}[itype]
    g = torch.Generator().manual_seed(seed)
    expert = torch.randn(256, width, generator=g)
    oc = mo.RffCostOracle(expert, feature_dim=D, input_type=itype, bw_samples=4000, bw_quantile=0.1, lambda_b=0.3,
                          seed=seed)
    oc.fit_cost(expert[:128] + 0.3 * torch.randn(128, width, generator=g))
    return oc, expert


def cost_ref(oc, s, a, s2, disc, lam, thr, clamp, prec=None):
    """(cost, ipm, bonus) of linear_cost.py:111-152 in float64, on operands rounded to `prec` (None: exact)."""
    rnd = rounder(prec)
    x = oc.rff_input(s.float(), a.float(), s2.float())
    pre = rnd(x) @ rnd(oc.rff_weight).t() + oc.rff_bias.double()
    dot = (torch.cos(pre) * math.sqrt(2.0 / oc.feature_dim)) @ oc.w.double()
    disc = disc.double()
    if clamp:
        dot = dot.clamp(-1.0, 0.0)
        bonus = torch.clamp(disc / thr, max=1.0) * -1.0
    else:
        bonus = disc
    ipm = (1 - lam) * dot
    return ipm - lam * bonus, ipm, lam * bonus


# ---------------------------------------------------------------------------------------------------
# GPU: the step against both oracles


@pytest.mark.gpu
@pytest.mark.parametrize("E", BATCHES)
@pytest.mark.parametrize("cid,prec", STEP_PARAMS)
def test_step_matches_oracles(cid, prec, E):
    c = case_data(cid)
    eng = engine(cid, prec)
    s, a, member, steps = inputs(c, E)
    sd, ad, md = s.cuda(), a.cuda(), member.cuda()
    std = steps.clone().cuda()
    nxt, disc, done = eng.step(sd, ad, md, std)
    fwd = eng.forward(sd, ad)
    if c["N"] == 1:
        assert float(disc.abs().max()) == 0.0

    preds = reference_deltas(c, s, a)
    nxt_ref, steps_ref, done_ref, disc_ref = oracle_step(c, s, a, member, steps, preds)
    s_next, s_disc, s_delta = scales(c, preds, disc_ref)
    assert torch.equal(std.cpu().long(), steps_ref)
    # the stand-alone entry point: same deltas, another post kernel (no state rows: never the TMA one)
    assert_close(eng.discrepancy(sd, ad), disc, s_disc, rel=2e-6, what="disc (stand-alone)")
    if prec != "bf16":
        assert_close(nxt, nxt_ref, s_next, what="next_state")
        assert_close(fwd, preds, s_delta, what="delta")
        if c["N"] > 1:
            assert_close(disc, disc_ref, s_disc, what="disc")
    mism = (done.cpu().bool() != done_ref).numpy()
    if mism.any():
        assert (threshold_margin(c, nxt_ref)[mism] < REL).all(), "termination differs away from any threshold"
    if E > 1:
        assert 0 < int(done_ref.sum()) < E

    preds2 = rounded_deltas(c, s, a, prec)
    nxt2, _, _, disc2 = oracle_step(c, s, a, member, steps, preds2)
    rel2 = REL_ROUNDED[prec]
    assert_close(nxt, nxt2, s_next, rel=rel2, what="next_state (operand-rounded oracle)")
    assert_close(fwd, preds2, s_delta, rel=rel2, what="delta (operand-rounded oracle)")
    if c["N"] > 1:
        assert_close(disc, disc2, s_disc, rel=rel2, what="disc (operand-rounded oracle)")

    if E == 257 and c["S"] % 2 == 0:
        # rows 8-byte but not 16-byte aligned: the float2 post kernel instead of the TMA one, same results
        buf = torch.zeros(2, E * c["S"] + 2, device="cuda")
        s8 = buf[0, 2:].view(E, c["S"])
        n8 = buf[1, 2:].view(E, c["S"])
        s8.copy_(sd)
        assert s8.data_ptr() % 16 == 8
        st8 = steps.clone().cuda()
        _, disc8, done8 = eng.step(s8, ad, md, st8, next_state=n8)
        assert torch.equal(n8, nxt) and torch.equal(done8, done) and torch.equal(st8, std)
        assert_close(disc8, disc, s_disc, rel=2e-6, what="disc (float2 post kernel)")

    if E == BATCHES[-1]:
        # three chunks of the workspace against one: step_cost stages the cost weights in chunk 0 only
        oc, _ = cost_oracle(c, "ss", 100)
        small = engine(cid, prec, chunk=CHUNK)
        assert math.ceil(E / CHUNK) == 3
        outs = []
        for e in (eng, small):
            e.load_rff(oc.rff_weight, oc.rff_bias, split=True, input_type="ss")
            st = steps.clone().cuda()
            outs.append(e.step_cost(sd, ad, md, st, oc.w.cuda(), 0.3, 0.5) + (st,))
        for x, y in zip(*outs):
            assert torch.equal(x, y)
        assert torch.equal(small.step(sd, ad, md, steps.clone().cuda())[0], nxt)


# ---------------------------------------------------------------------------------------------------
# GPU: the fused step cost for every input type


class _FixedDisc:
    def __init__(self, disc, threshold):
        self.disc, self.threshold = disc, threshold

    def get_action_discrepancy(self, states, actions):
        return self.disc.clone()


class _Ensemble:
    """What VecSimEnv reads of a DynamicsEnsemble."""

    def __init__(self, eng):
        self.eng, self.state_dim, self.action_dim, self.num_models = eng, eng.S, eng.A, eng.N

    def engine(self):
        return self.eng


def check_step_cost(cid, prec, itype, split, D, E=257):
    from amp_extensions_b200 import RBFLinearCost
    from amp_extensions_b200.sim_env import VecSimEnv
    c = case_data(cid)
    eng = engine(cid, prec)
    oc, expert = cost_oracle(c, itype, D)
    cost = RBFLinearCost(expert, feature_dim=D, input_type=itype, bw_samples=4000, bw_quantile=0.1, lambda_b=0.3,
                         seed=7, precision=prec, split=split)
    assert torch.equal(cost.rff.weight.data, oc.rff_weight) and torch.equal(cost.rff.bias.data, oc.rff_bias)
    cost.w = oc.w.clone()
    VecSimEnv(_Ensemble(eng), 4, termination=termination(c), cost=cost)   # attach_cost loads the layer
    assert eng.rff_split == split
    s, a, member, steps = inputs(c, E, seed=3)
    sd, ad, md, w = s.cuda(), a.cuda(), member.cuda(), oc.w.cuda()
    # a threshold inside the discrepancy's range: both sides of min(disc / threshold, 1)
    thr = max(float(eng.discrepancy(sd, ad).median()), 1e-6)
    for lam, clamp in ((0.0, True), (0.3, True), (1.0, True), (0.3, False)):
        nxt, disc, done, cst, ipm, bonus = eng.step_cost(sd, ad, md, steps.clone().cuda(), w, lam, thr,
                                                         clamp_cost=clamp)
        # the cost of the step's own s' and discrepancy (both are checked against the oracles above)
        s2 = nxt.cpu()
        ref = cost_ref(oc, s, a, s2, disc.cpu(), lam, thr, clamp, None if split else prec)
        cs = max(float(ref[0].abs().max()), 1e-6)
        for got, want, name in zip((cst, ipm, bonus), ref, ("cost", "ipm", "bonus")):
            assert_close(got, want, cs, what=f"{name} (lambda_b {lam}, clamp {clamp})")
        assert torch.equal(cst, ipm - bonus)
        # the same cost through RBFLinearCost's own engine (rows built on the host by input_type)
        cost.lambda_b = lam
        cost.cost_range = [-1.0, 0.0] if clamp else None
        own, info = cost.get_bonus_costs(s, a, _FixedDisc(disc.cpu(), thr), next_states=s2)
        assert_close(cst, own[:, 0], cs, rel=1e-4, what=f"fused vs RBFLinearCost.get_bonus_costs ({itype})")


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["tf32", "fp16"])
@pytest.mark.parametrize("cid", list(COST_CASES))
@pytest.mark.parametrize("split", [True, False])
@pytest.mark.parametrize("itype", INPUT_TYPES)
def test_step_cost_matches_oracle(itype, split, cid, prec):
    check_step_cost(cid, prec, itype, split, COST_CASES[cid])


@pytest.mark.gpu
@pytest.mark.parametrize("cid", ["n6_s2mod4", "n7_odd"])
def test_unaligned_rows(cid):
    """State and next-state rows 4 bytes past an 8-byte boundary (scalar post kernel, non-vector prep, unfused cost
    rows) and 8 bytes past a 16-byte one (float2 post kernel): the aligned run's results."""
    c = case_data(cid)
    eng = engine(cid, "fp16")
    oc, _ = cost_oracle(c, "ss", 100)
    eng.load_rff(oc.rff_weight, oc.rff_bias, split=True, input_type="ss")
    E, S = 1029, c["S"]
    s, a, member, steps = inputs(c, E, seed=5)
    ad, md, w = a.cuda(), member.cuda(), oc.w.cuda()
    st0 = steps.clone().cuda()
    al = eng.step_cost(s.cuda(), ad, md, st0, w, 0.3, 0.5)
    for off in (1, 2):   # floats
        buf = torch.zeros(2, E * S + 4, device="cuda")
        sv, nv = buf[0, off:off + E * S].view(E, S), buf[1, off:off + E * S].view(E, S)
        sv.copy_(s.cuda())
        assert sv.data_ptr() % 16 == 4 * off
        st = steps.clone().cuda()
        out = eng.step_cost(sv, ad, md, st, w, 0.3, 0.5, next_state=nv)
        assert torch.equal(out[0], al[0]) and torch.equal(out[2], al[2]) and torch.equal(st, st0)
        assert_close(out[1], al[1], al[1].mean().item(), rel=2e-6, what="disc")
        assert_close(out[3], al[3], al[3].abs().max().item(), rel=1e-5, what="cost")


@pytest.mark.gpu
def test_state_dim_over_post_limit():
    """S = 257: the forward pass (the only shape with a two-tile final layer, SP = 512) matches both oracles; the post
    kernel's S <= 256 limit is refused on the host with a clean error and the handle stays usable."""
    from amp_extensions_b200._lib import SimstepError
    from amp_extensions_b200.engine import Engine
    S, A, N, hidden = 257, 8, 2, [64]
    c = dict(S=S, A=A, N=N, hidden=hidden, dense=True, act="relu", transform=True, humanoid=False)
    c["ws"], c["bs"] = mo.init_ensemble(S, A, hidden, N, dense_connect=True, base_seed=5)
    c["tf"] = mo.get_transformations(*H.synth_dataset(1024, S, A, 5))
    eng = Engine(S, A, N, hidden, dense_connect=True, activation="relu", transform=True, precision="fp16")
    eng.load_ensemble(c["ws"], c["bs"], c["tf"])
    s, a, member, steps = inputs(c, 300)
    sd, ad = s.cuda(), a.cuda()
    fwd = eng.forward(sd, ad)
    ref = reference_deltas(c, s, a)
    s_delta = float(ref.abs().max())
    assert_close(fwd, ref, s_delta, what="delta")
    assert_close(fwd, rounded_deltas(c, s, a, "fp16"), s_delta, rel=REL_ROUNDED["fp16"], what="delta (operand-rounded)")
    oc, _ = cost_oracle(c, "ss", 100)
    eng.load_rff(oc.rff_weight, oc.rff_bias, split=True, input_type="ss")
    for call in (lambda: eng.step(sd, ad, member.cuda(), steps.cuda()),
                 lambda: eng.discrepancy(sd, ad),
                 lambda: eng.step_cost(sd, ad, member.cuda(), steps.cuda(), oc.w.cuda(), 0.3, 0.5)):
        with pytest.raises(SimstepError, match="state_dim > 256"):
            call()
        assert torch.equal(eng.forward(sd, ad), fwd)


@pytest.mark.gpu
def test_ambiguous_rff_width_is_refused():
    """An untyped load cannot tell 'sa' from 'ss' when S == A, nor 's' from 'sa' when A == 0: it is refused, and the
    typed load gives each type's oracle cost."""
    from amp_extensions_b200._lib import SimstepError
    for cid, types, dim in (("square", ("sa", "ss"), lambda c: 2 * c["S"]), ("a0", ("s", "sa"), lambda c: c["S"])):
        c = case_data(cid)
        eng = engine(cid, "tf32")
        oc, _ = cost_oracle(c, types[0], 100)
        assert oc.rff_weight.shape[1] == dim(c)
        with pytest.raises(SimstepError, match="more than one input_type"):
            eng.load_rff(oc.rff_weight, oc.rff_bias, split=True)
        for t in types:
            check_step_cost(cid, "tf32", t, True, 100, E=64)


# ---------------------------------------------------------------------------------------------------
# GPU: both forward paths and the guard zones at every shape (the switches are read once per process)

MATRIX_SCRIPT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "write_matrix_outputs.py")


def run_matrix(tmp_path, name, **env_over):
    out = str(tmp_path / f"{name}.npz")
    env = {k: v for k, v in os.environ.items() if k not in ("SIMSTEP_CHAIN", "SIMSTEP_DEBUG_GUARDS")}
    env.update(env_over)
    res = subprocess.run([sys.executable, MATRIX_SCRIPT, out], env=env, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-3000:]
    return np.load(out)


@pytest.mark.gpu
def test_every_shape_matches_one_launch_per_layer_bit_for_bit(tmp_path):
    default, per_layer = run_matrix(tmp_path, "default"), run_matrix(tmp_path, "per_layer", SIMSTEP_CHAIN="0")
    assert sorted(default.files) == sorted(per_layer.files)
    for k in default.files:
        if not k.startswith("launches_"):
            assert np.array_equal(default[k], per_layer[k], equal_nan=True), k
    for c in CASES:
        for prec in ("tf32", "fp16"):
            want = len(c["hidden"]) + 1
            assert (per_layer[f"launches_{c['id']}_{prec}"] == want).all()
            # the restatement of chain_ok: every case with a hidden layer takes the column-fused kernel
            assert (default[f"launches_{c['id']}_{prec}"] == (1 if chain_taken(len(c["hidden"])) else want)).all()


@pytest.mark.gpu
def test_guard_zones_stay_intact_at_every_shape(tmp_path):
    out = run_matrix(tmp_path, "guards", SIMSTEP_DEBUG_GUARDS="1")
    for c in CASES:
        for prec in ("tf32", "fp16"):
            n, bad = out[f"guards_{c['id']}_{prec}"]
            assert n >= 3 and bad == 0, (c["id"], prec, n, bad)   # x, deltas, cost rows (+ activations)


# ---------------------------------------------------------------------------------------------------
# CPU: the dispatch predicates of csrc/api.cu, and the oracles themselves

K_POST_MAX_ELEMS = 256            # elementwise.cuh kPostMaxElems
K_CHAIN_MAX_LAYERS = 8 + 1        # gemm_chain.cuh kChainMaxLayers = SIMSTEP_MAX_HIDDEN + 1


def post_tma_plan_ok(S, N):
    """post_tma.cuh post_tma_plan(S, DP, NM).ok with DP = round_up(S, 4) (api.cu simstep_create)."""
    DP = (S + 3) // 4 * 4
    stage = 2 * S * 4 + N * 2 * DP * 4
    rings, stages, budget = 20 // 2, 2, 216 * 1024
    while rings * stages * stage > budget and rings > 1:
        rings -= 1
    return S % 2 == 0 and S <= K_POST_MAX_ELEMS and DP % 4 == 0 and rings * stages * stage <= budget


def chain_taken(L):
    """api.cu chain_ok: L >= 1 and L + 1 <= kChainMaxLayers (the L2 working-set test holds at every shape here)."""
    return L >= 1 and L + 1 <= K_CHAIN_MAX_LAYERS


def step_branches(c, prec, align, itype=None):
    """The launch paths one step (itype None) or step_cost of case c takes with state rows `align` bytes aligned, as
    (what, variant) tuples."""
    S, A, N = c["S"], c["A"], c["N"]
    b = set()
    # api.cu launch_prep: vec = S, A even and 8-byte aligned sources
    b.add(("prep", "vec" if S % 2 == 0 and A % 2 == 0 and align % 8 == 0 else "scalar",
           "transform" if c["transform"] else "no transform"))
    b.add(("forward", "chain" if chain_taken(len(c["hidden"])) else "per layer"))
    # api.cu simstep_step_cost: fuse = input_type 'ss' with float2-able rows
    fuse = itype == "ss" and S % 2 == 0 and align % 8 == 0
    # api.cu launch_post: vec2 (even S, 8-byte rows), tma (plan ok, vec2, 16-byte state), the NM switch
    vec2 = S % 2 == 0 and align % 8 == 0
    if post_tma_plan_ok(S, N) and vec2 and align % 16 == 0:
        b.add(("post tma", N))
        b.add(("post tma S", 226 if S == 226 else 0))              # the S = 226 specialisation
        # the ElemF16 instantiation unless the kernel stores tf32 or bf16 cost rows
        b.add(("post tma cost rows", prec if fuse else None))
    else:
        b.add(("post float2" if vec2 else "post scalar", N))
    if itype is not None:
        # api.cu rff_sources: one branch per input_type, unless the post kernel wrote the rows itself
        b.add(("cost rows", "fused post store", prec) if fuse else ("cost rows", "rff_pack " + itype, prec))
    return b


def suite_runs():
    """(case, precision, row alignment, input_type) of every step the GPU tests above run."""
    runs = []
    for cid, prec in STEP_PARAMS:
        c = CASE[cid]
        runs.append((c, prec, 16, None))                    # test_step_matches_oracles
        if c["S"] % 2 == 0:
            runs.append((c, prec, 8, None))                 # its float2 variant
        runs.append((c, prec, 16, "ss"))                    # its chunked step_cost
    for cid in COST_CASES:
        for prec in ("tf32", "fp16"):
            for t in INPUT_TYPES:
                runs.append((CASE[cid], prec, 16, t))       # test_step_cost_matches_oracle
    for cid in ("n6_s2mod4", "n7_odd"):
        for align in (16, 4, 8):
            runs.append((CASE[cid], "fp16", align, "ss"))   # test_unaligned_rows
    for t in ("s", "sa"):
        runs.append((CASE["a0"], "tf32", 16, t))            # test_ambiguous_rff_width_is_refused
    return runs


def test_case_table_reaches_every_step_branch():
    reached = set()
    for c, prec, align, itype in suite_runs():
        reached |= step_branches(c, prec, align, itype)
    precs = ("tf32", "fp16", "bf16")
    required = {("post tma", nm) for nm in range(1, 9)} | {("post float2", nm) for nm in range(1, 9)}
    required |= {("post tma S", 226), ("post tma S", 0)} | {("post tma cost rows", p) for p in precs + (None,)}
    required |= {("prep", "vec", "transform"), ("prep", "scalar", "transform"), ("prep", "vec", "no transform")}
    required |= {("forward", "chain"), ("forward", "per layer")}
    required |= {("cost rows", "rff_pack " + t, p) for t in INPUT_TYPES for p in ("tf32", "fp16")}
    required |= {("cost rows", "rff_pack ss", "bf16")} | {("cost rows", "fused post store", p) for p in precs}
    assert any(b[0] == "post scalar" for b in reached)
    missing = required - reached
    for b in sorted(reached, key=str):
        print("reached:", *b)
    assert not missing, f"branches no case reaches: {sorted(missing, key=str)}"
    for c in CASES:
        assert c["covers"]
        assert len(c["hidden"]) <= 8 and c["N"] <= 8


def test_operand_rounded_oracle_is_the_reference_oracle_without_rounding():
    c = case_data("n7_odd")
    s, a, _, _ = inputs(c, 64)
    ref = reference_deltas(c, s, a)
    assert torch.equal(rounded_deltas(c, s, a, None), ref)
    scale = float(ref.abs().max())
    err = {p: rel_err(rounded_deltas(c, s, a, p), ref, scale) for p in ("tf32", "fp16", "bf16")}
    # the operand error itself: 10 explicit mantissa bits for tf32 and fp16, 7 for bf16 (about 8x more)
    assert 1e-5 < err["tf32"] < REL and 1e-5 < err["fp16"] < REL
    assert err["bf16"] > 3 * err["fp16"]
    c2 = case_data("no_transform")
    s2, a2, _, _ = inputs(c2, 16)
    assert torch.equal(rounded_deltas(c2, s2, a2, None), reference_deltas(c2, s2, a2))
