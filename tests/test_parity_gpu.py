"""GPU parity of the CUDA path (through the C ABI) against the reference's golden vectors and the oracle.

Tolerance (BASELINE.json north_star): 1e-3 relative for next-state and reward against the fp32 reference,
tensor-core operands with >= 10 mantissa bits (tf32 or fp16) and fp32 accumulation.  "Relative" is taken
per element against max(|ref|, scale) where scale is the typical magnitude of that output (element-wise
relative error is ill-posed at zero crossings); each test states its scale.  Termination masks must be
identical except for rows whose margin to a threshold is inside that tolerance.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import milo_oracle as mo
from tests import helpers as H

pytestmark = pytest.mark.gpu

REL = 1e-3
PRECISIONS = ["tf32", "fp16"]


def assert_close(x, ref, scale, rel=REL, what=""):
    x, ref = x.detach().double().cpu(), ref.detach().double().cpu()
    tol = rel * torch.maximum(ref.abs(), torch.as_tensor(scale, dtype=torch.float64).expand_as(ref))
    bad = (x - ref).abs() > tol
    assert torch.isfinite(x).all(), f"{what}: non-finite output"
    l2 = float((x - ref).norm() / ref.norm().clamp_min(1e-300))   # the plain relative L2 error, for the record
    assert not bad.any(), (f"{what}: {int(bad.sum())} of {bad.numel()} outside {rel:g} relative; worst abs err "
                           f"{float((x - ref).abs().max()):.3e} at ref {float(ref.flatten()[(x - ref).abs().argmax()]):.3e}; "
                           f"relative L2 {l2:.3e}")


def make_engine(case, precision, **kw):
    from amp_extensions_b200.engine import Engine
    eng = Engine(case["S"], case["A"], case["N"], case["hidden"], dense_connect=case["dense"],
                 activation=case["act"], transform=True, precision=precision, **kw)
    eng.load_ensemble(case["ws"], case["bs"], case["tf"])
    return eng


# ---------------------------------------------------------------------------------------------------
# the GEMM kernel alone

@pytest.mark.parametrize("prec", ["tf32", "fp16", "bf16"])
@pytest.mark.parametrize("shape", [(1, 1, 8, 8), (1, 128, 256, 64), (2, 129, 257, 100), (4, 1000, 226, 2302),
                                   (3, 5000, 512, 1278)])
def test_debug_gemm_matches_fp64(prec, shape):
    from amp_extensions_b200 import _lib
    lib = _lib.load()
    groups, m, n, k = shape
    g = torch.Generator(device="cuda").manual_seed(m * 7 + n)
    a = torch.randn(groups, m, k, device="cuda", generator=g)
    b = torch.randn(groups, n, k, device="cuda", generator=g) / k ** 0.5
    bias = torch.randn(groups, n, device="cuda", generator=g)
    d = torch.full((groups, m, n), float("nan"), device="cuda")
    rc = lib.simstep_debug_gemm(_lib.PREC[prec], groups, m, n, k, C.c_void_p(a.data_ptr()), C.c_void_p(b.data_ptr()),
                                C.c_void_p(bias.data_ptr()), C.c_void_p(d.data_ptr()), None)
    _lib.check(rc)

    def rnd(x):
        if prec == "tf32":
            return ((x.contiguous().view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32)
        return x.half().float() if prec == "fp16" else x.bfloat16().float()

    ref = torch.einsum("gmk,gnk->gmn", rnd(a).double(), rnd(b).double()) + bias.double()[:, None, :]
    # operands are rounded identically on both sides, so only the fp32 accumulation order differs
    assert (d.double() - ref).abs().max().item() <= 3e-5 * max(1.0, (k / 256) ** 0.5) * ref.abs().max().item()


# ---------------------------------------------------------------------------------------------------
# ensemble forward / discrepancy against the reference's own outputs

@pytest.mark.parametrize("prec", PRECISIONS)
@pytest.mark.parametrize("tag", ["tiny_dense", "tiny_plain_tanh"])
def test_tiny_forward_matches_reference(tag, prec):
    c = H.tiny_case(tag)
    eng = make_engine(c, prec)
    preds = eng.forward(c["xs"], c["xa"])
    scale = c["tf"][5].abs().max().item()  # diff_scale: the unit the network's output is expressed in
    assert_close(preds, c["preds"], scale, what="delta")
    disc = eng.discrepancy(c["xs"], c["xa"])
    assert_close(disc, c["disc"], c["disc"].mean().item(), what="disc")


@pytest.mark.parametrize("prec", PRECISIONS)
def test_north_star_forward_matches_reference(prec):
    c = H.ns_case()
    eng = make_engine(c, prec)
    preds = eng.forward(c["xs"], c["xa"])
    assert_close(preds, c["preds"], c["tf"][5].abs().max().item(), what="delta")
    rel_l2 = ((preds.cpu() - c["preds"]).norm() / c["preds"].norm()).item()
    assert rel_l2 < REL
    assert_close(eng.discrepancy(c["xs"], c["xa"]), c["disc"], c["disc"].mean().item(), what="disc")


def test_bf16_operands_miss_the_tolerance_budget():
    """Why the default operand format is fp16 and not bf16: measured, not assumed (SURVEY.md section 7)."""
    c = H.ns_case()
    e16, eb = make_engine(c, "fp16"), make_engine(c, "bf16")
    err16 = ((e16.forward(c["xs"], c["xa"]).cpu() - c["preds"]).norm() / c["preds"].norm()).item()
    errb = ((eb.forward(c["xs"], c["xa"]).cpu() - c["preds"]).norm() / c["preds"].norm()).item()
    assert err16 < REL and errb > 3 * err16


@pytest.mark.parametrize("prec", PRECISIONS)
def test_threshold_matches_reference(prec):
    from amp_extensions_b200 import AmpDataset, DynamicsEnsemble
    c = H.ns_case()
    s, a, s2 = H.synth_dataset(8192, 226, 28, 0)
    n = c["threshold_rows"]
    full = AmpDataset(s, a, s2)
    ens = DynamicsEnsemble(226, 28, full, None, num_models=4, hidden_sizes=[512] * 4, dense_connect=True,
                           transform=True, base_seed=100, precision=prec)
    for tf_mine, tf_ref in zip(ens.transformations, c["tf"]):
        assert torch.equal(tf_mine, tf_ref)
    for k in range(4):  # same seed, same init order as the reference (dynamics.py:184-196)
        for l, lin in enumerate(ens.models[k].model.fc_layers):
            assert torch.equal(lin.weight.data, c["ws"][k][l]) and torch.equal(lin.bias.data, c["bs"][k][l])
    ens.train_dataset = AmpDataset(s[:n], a[:n], s2[:n])
    ens.compute_threshold()
    assert ens.threshold == pytest.approx(c["threshold"], rel=REL)


# ---------------------------------------------------------------------------------------------------
# the env step: next state, discrepancy, termination, counters

def oracle_step(c, s, a, member, steps, **kw):
    preds = mo.ensemble_forward(c["ws"], c["bs"], c["tf"], s, a, c["dense"], c["act"])
    active = preds[member.long(), torch.arange(s.shape[0])]
    nxt, st, done = mo.simenv_step(s.double().numpy(), active.numpy(), steps.numpy(), **kw)
    return preds, torch.from_numpy(nxt), torch.from_numpy(st), torch.from_numpy(done), mo.discrepancy_from_preds(preds)


def collision_margin(ob):
    """Smallest distance of any tested quantity to its threshold (sim_env.py:188, 236), per row."""
    ob = np.asarray(ob, dtype=np.float64)
    m = np.full(ob.shape[0], np.inf)
    for body in mo.HUMANOID3D_FALL_BODIES:
        shape, p0, p1 = mo.HUMANOID3D_BODY_DEFS[body]
        off = 9 * body + 1
        y = ob[:, 0] + ob[:, off + 1]
        lim = 0.5 * p0 + 1e-4
        if shape == "sphere":
            m = np.minimum(m, np.abs(y - lim))
        else:
            cap = 0.5 * p1 * ob[:, off + 4]
            m = np.minimum(m, np.minimum(np.abs(y + cap - lim), np.abs(y - cap - lim)))
    return m


@pytest.mark.parametrize("prec", PRECISIONS)
@pytest.mark.parametrize("E", [1, 127, 128, 129, 1024])
def test_step_matches_oracle(prec, E):
    from amp_extensions_b200.engine import HumanoidTermination
    c = H.ns_case()
    eng = make_engine(c, prec)
    eng.set_termination(HumanoidTermination(horizon=300, enable_velocity_check=True))
    s = H.humanoid_like_states(E, seed=11)
    g = torch.Generator().manual_seed(12)
    a = torch.randn(E, 28, generator=g)
    member = torch.randint(0, 4, (E,), generator=g, dtype=torch.int32)
    steps = torch.randint(0, 300, (E,), generator=g, dtype=torch.int32)
    steps[: max(1, E // 8)] = 299
    _, nxt_ref, steps_ref, done_ref, disc_ref = oracle_step(c, s, a, member, steps, horizon=300,
                                                            enable_velocity_check=True)
    sd, ad = s.cuda(), a.cuda()
    md, std = member.cuda(), steps.clone().cuda()
    nxt, disc, done = eng.step(sd, ad, md, std)
    # scale of a state element: the dataset's per-dimension spread (state_scale of the transforms)
    assert_close(nxt, nxt_ref, c["tf"][1].mean().item(), what="next_state")
    assert_close(disc, disc_ref, disc_ref.mean().item(), what="disc")
    assert torch.equal(std.cpu(), steps_ref.to(torch.int32))
    mism = done.cpu().bool() != done_ref
    if mism.any():
        margin = np.minimum(collision_margin(nxt_ref.numpy()), np.abs(np.abs(nxt_ref.numpy()[:, 136:]) - 100).min(1))
        assert (margin[mism.numpy()] < REL * 1.0).all(), "termination mask differs away from any threshold"
    assert 0 < int(done_ref.sum()) < E or E == 1  # the inputs exercise both outcomes


@pytest.mark.parametrize("prec", PRECISIONS)
def test_step_in_place_and_optional_outputs(prec):
    c = H.tiny_case("tiny_dense")
    eng = make_engine(c, prec)
    g = torch.Generator().manual_seed(3)
    s, a = torch.randn(300, 20, generator=g).cuda(), torch.randn(300, 6, generator=g).cuda()
    member = torch.zeros(300, dtype=torch.int32, device="cuda")
    steps = torch.zeros(300, dtype=torch.int32, device="cuda")
    ref_next, ref_disc, _ = eng.step(s, a, member, steps.clone())
    s2 = s.clone()
    out, disc, done = eng.step(s2, a, member, steps, next_state=s2, want_disc=False, want_done=False)
    assert out.data_ptr() == s2.data_ptr() and disc is None and done is None
    assert torch.equal(s2, ref_next)  # aliasing next_state with state is allowed (sim_env.py:158 is in place)
    assert int(steps.min()) == 1 and int(steps.max()) == 1


def test_empty_batch_is_a_no_op():
    c = H.tiny_case("tiny_dense")
    eng = make_engine(c, "tf32")
    assert eng.forward(torch.zeros(0, 20), torch.zeros(0, 6)).shape == (3, 0, 20)
    assert eng.discrepancy(torch.zeros(0, 20), torch.zeros(0, 6)).shape == (0,)


def test_identical_members_have_zero_discrepancy():
    c = dict(H.tiny_case("tiny_dense"))
    c["ws"] = [c["ws"][0]] * c["N"]
    c["bs"] = [c["bs"][0]] * c["N"]
    eng = make_engine(c, "fp16")
    assert float(eng.discrepancy(c["xs"], c["xa"]).abs().max()) == 0.0


@pytest.mark.parametrize("prec", PRECISIONS)
def test_rows_are_independent_and_chunking_is_invisible(prec):
    """Full-size properties (40 000 rows, BASELINE.json config 2): a row's result does not depend on the
    batch around it, on its position, or on how the library chunks the batch."""
    c = H.ns_case()
    E = 40000
    g = torch.Generator().manual_seed(21)
    s, a = torch.randn(E, 226, generator=g).cuda(), torch.randn(E, 28, generator=g).cuda()
    big = make_engine(c, prec)
    d_all = big.discrepancy(s, a)
    assert torch.isfinite(d_all).all()
    perm = torch.randperm(E, generator=g).cuda()
    assert torch.equal(big.discrepancy(s[perm], a[perm]), d_all[perm])
    assert torch.equal(big.discrepancy(s[1000:1777], a[1000:1777]), d_all[1000:1777])
    small = make_engine(c, prec, max_chunk_envs=4096)
    assert torch.equal(small.discrepancy(s, a), d_all)
    # forward and discrepancy come from the same pass: recompute the norm from the returned deltas
    f = big.forward(s[:4096], a[:4096]).double()
    pair = torch.stack([(f[i] - f[j]).norm(dim=1) for i in range(4) for j in range(i + 1, 4)]).max(0).values
    assert_close(d_all[:4096], pair, pair.mean().item(), rel=1e-5, what="disc vs forward")


@pytest.mark.parametrize("prec", PRECISIONS)
def test_extreme_inputs_stay_finite_or_propagate_nan(prec):
    c = H.tiny_case("tiny_dense")
    eng = make_engine(c, prec)
    s, a = c["xs"].clone(), c["xa"].clone()
    s[0] = 1e6   # an exploded state: fp16 operands saturate instead of overflowing
    s[1, 3] = float("nan")
    out = eng.forward(s, a).cpu()
    assert torch.isfinite(out[:, 0]).all()
    assert torch.isnan(out[:, 1]).any()
    assert torch.isfinite(out[:, 2:]).all()
    assert torch.isnan(eng.discrepancy(s, a).cpu()[1])


# ---------------------------------------------------------------------------------------------------
# MILO cost

@pytest.mark.parametrize("prec", PRECISIONS)
@pytest.mark.parametrize("tag,D", [("cost64", 64), ("cost512", 512)])
def test_rbf_linear_cost_matches_reference(tag, D, prec):
    from amp_extensions_b200 import RBFLinearCost
    g = H.golden()
    c = H.ns_case()
    cost = RBFLinearCost(H.ns_expert(), feature_dim=D, input_type="ss", bw_quantile=0.1, lambda_b=0.0025, seed=100,
                         precision=prec)
    assert cost.bw == float(g[f"{tag}/bw"])  # host-side fit: same RNG stream, same arithmetic
    wsum = g[f"{tag}/rff_wsum"]
    assert float(cost.rff.weight.data.double().sum()) == wsum[0] and float(cost.rff.bias.data.double().sum()) == wsum[1]
    phi_scale = (2.0 / D) ** 0.5
    assert_close(cost.phi_e, H.t(g[f"{tag}/phi_e"]), phi_scale, what="phi_e")
    nxt = H.t(g[f"{tag}/next"])
    pi = torch.cat([c["xs"], nxt], dim=1)
    assert_close(cost.get_rep(pi), H.t(g[f"{tag}/rep"]), phi_scale, what="rep")
    mmd = cost.fit_cost(pi)
    assert mmd == pytest.approx(float(g[f"{tag}/mmd"]), rel=REL)
    w_ref = H.t(g[f"{tag}/w"])
    assert_close(cost.w, w_ref, w_ref.abs().max().item(), what="w")
    cost.w = w_ref.clone()  # isolate the remaining checks from the fit
    costs_ref = H.t(g[f"{tag}/costs"])
    cscale = max(costs_ref.abs().max().item(), 1e-6)
    assert_close(cost.get_costs(pi), costs_ref, cscale, what="costs")
    ec = cost.get_expert_cost()                               # linear_cost.py:105-109, evaluated on the device
    assert ec.dim() == 0 and abs(float(ec) - float(g[f"{tag}/expert_cost"])) <= REL * max(cscale, abs(float(g[f"{tag}/expert_cost"])))

    class Ens:  # the reference passes the ensemble object (linear_cost.py:132)
        threshold = c["threshold"]

        @staticmethod
        def get_action_discrepancy(s, a):
            return c["disc"]

    total, info = cost.get_bonus_costs(c["xs"], c["xa"], Ens, next_states=nxt)
    assert total.shape == (48, 1)
    tot_ref = H.t(g[f"{tag}/total"])
    assert_close(total, tot_ref, tot_ref.abs().max().item(), what="total cost")
    for k in ("bonus", "ipm", "v_targ", "cost"):
        ref = H.t(g[f"{tag}/info_{k}"])
        assert_close(info[k], ref, max(ref.abs().max().item(), 1e-6), what=k)


@pytest.mark.parametrize("prec", PRECISIONS)
def test_fused_step_cost_matches_oracle(prec):
    """BASELINE.json config 2 path: step + discrepancy bonus + IPM cost in one call."""
    from amp_extensions_b200 import RBFLinearCost
    from amp_extensions_b200.engine import HumanoidTermination
    c = H.ns_case()
    E = 2000
    s = H.humanoid_like_states(E, seed=31)
    g = torch.Generator().manual_seed(32)
    a = torch.randn(E, 28, generator=g)
    member = torch.randint(0, 4, (E,), generator=g, dtype=torch.int32)
    steps = torch.zeros(E, dtype=torch.int32)
    lam, thr = 0.0025, c["threshold"]
    oc = mo.RffCostOracle(H.ns_expert(), feature_dim=512, input_type="ss", bw_quantile=0.1, lambda_b=lam, seed=100)
    _, nxt_ref, _, done_ref, disc_ref = oracle_step(c, s, a, member, steps)
    oc.fit_cost(torch.cat([s, nxt_ref.float()], dim=1)[:1024])
    cost_ref, info_ref = oc.get_bonus_costs(s, a, disc_ref, thr, next_states=nxt_ref.float())

    eng = make_engine(c, prec)
    eng.set_termination(HumanoidTermination())
    eng.load_rff(oc.rff_weight, oc.rff_bias, split=True)
    nxt, disc, done, cost, ipm, bonus = eng.step_cost(s.cuda(), a.cuda(), member.cuda(), steps.cuda(), oc.w.cuda(),
                                                       lam, thr)
    assert_close(nxt, nxt_ref, c["tf"][1].mean().item(), what="next_state")
    assert_close(disc, disc_ref, disc_ref.mean().item(), what="disc")
    cs = cost_ref.abs().max().item()
    assert_close(cost, cost_ref[:, 0], cs, what="cost")
    assert_close(ipm, info_ref["ipm"][:, 0], cs, what="ipm")
    assert_close(bonus, info_ref["bonus"][:, 0], info_ref["bonus"].abs().max().item(), what="bonus")
    # reward = -cost (batch_reinforce.py:144) at 1e-3 of the reward scale
    assert_close(-cost, -cost_ref[:, 0], cs, what="reward")
    # cost_range=None variant (linear_cost.py:103, 137-138)
    oc.cost_range = None
    cost_ref2, _ = oc.get_bonus_costs(s, a, disc_ref, thr, next_states=nxt_ref.float())
    out = eng.step_cost(s.cuda(), a.cuda(), member.cuda(), steps.cuda(), oc.w.cuda(), lam, 1.0, 0.0, 0.0, False)
    assert_close(out[3], cost_ref2[:, 0], cost_ref2.abs().max().item(), what="unclamped cost")


# ---------------------------------------------------------------------------------------------------
# BASELINE.json configs[4]: the 8-member, hidden 1024 x 4 ensemble


def test_scale_config_8x1024_matches_oracle():
    """8 x (1024 x 4) dense-connect members (28 discrepancy pairs, K up to 4350): step + discrepancy against the
    fp32 oracle on the same seed-generated weights, odd batch so the row-pair staging sees a trailing row."""
    from amp_extensions_b200.engine import Engine, HumanoidTermination
    S, A, N, hidden, E = 226, 28, 8, [1024] * 4, 257
    ws, bs = mo.init_ensemble(S, A, hidden, N, dense_connect=True, base_seed=100)
    s_d, a_d, s2_d = H.synth_dataset(4096, S, A, 0)
    tf = mo.get_transformations(s_d, a_d, s2_d)
    eng = Engine(S, A, N, hidden, dense_connect=True, activation="relu", transform=True, precision="fp16")
    eng.load_ensemble(ws, bs, tf)
    eng.set_termination(HumanoidTermination(horizon=300))
    s = H.humanoid_like_states(E, seed=21)
    g = torch.Generator().manual_seed(22)
    a = torch.randn(E, A, generator=g)
    member = torch.randint(0, N, (E,), generator=g, dtype=torch.int32)
    steps = torch.zeros(E, dtype=torch.int32)
    preds = mo.ensemble_forward(ws, bs, tf, s, a)
    active = preds[member.long(), torch.arange(E)]
    nxt_ref, _, done_ref = mo.simenv_step(s.double().numpy(), active.numpy(), steps.numpy())
    disc_ref = mo.discrepancy_from_preds(preds)
    nxt, disc, done = eng.step(s.cuda(), a.cuda(), member.cuda(), steps.cuda())
    assert_close(nxt, torch.from_numpy(nxt_ref), tf[1].mean().item(), what="next_state")
    assert_close(disc, disc_ref, disc_ref.mean().item(), what="disc")
    mism = done.cpu().bool().numpy() != done_ref
    if mism.any():
        assert (collision_margin(nxt_ref)[mism] < REL).all()
    fwd = eng.forward(s[:64], a[:64])
    assert_close(fwd, preds[:, :64], tf[5].abs().max().item(), what="delta")


# ---------------------------------------------------------------------------------------------------
# MLPCost (linear_cost.py:154-301): MLP features through the grouped GEMM + tanh/cos head


class _FixedDiscEnsemble:
    def __init__(self, disc, threshold):
        self.disc, self.threshold = disc, threshold

    def get_action_discrepancy(self, states, actions):
        return self.disc.clone()


@pytest.mark.parametrize("prec", PRECISIONS)
@pytest.mark.parametrize("tag", ["two_hidden", "one_hidden_quirk", "three_tanh"])
def test_mlp_cost_matches_reference(tag, prec):
    """Same seed -> the same net as the reference (bit for bit, built on the host); features, fitted weights,
    costs and the bonus combine against the reference's own outputs.  Scale of a feature: sqrt(2/D)."""
    import os
    from amp_extensions_b200 import MLPCost
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "mlpcost_golden.npz"))
    expert = torch.from_numpy(g["expert"])
    D = int(g[f"{tag}/feature_dim"])
    cost = MLPCost(expert, hidden_dims=g[f"{tag}/hidden"].tolist(), activation=str(g[f"{tag}/act"]), feature_dim=D,
                   input_type="ss", bw_quantile=0.1, lambda_b=0.3, seed=100, precision=prec)
    lin = cost._linears()
    assert len(lin) == int(g[f"{tag}/n_linear"])
    for i, l in enumerate(lin):
        assert np.array_equal(l.weight.data.numpy(), g[f"{tag}/w{i}"])
    assert cost.bw == float(g[f"{tag}/bw"])
    xs, xa, nxt = (torch.from_numpy(g[k]) for k in ("xs", "xa", "next"))
    pi = torch.cat([xs, nxt], dim=1)
    fscale = (2.0 / g[f"{tag}/rep"].shape[1]) ** 0.5
    assert_close(cost.phi_e, torch.from_numpy(g[f"{tag}/phi_e"]), fscale, what="phi_e")
    assert_close(cost.get_rep(pi), torch.from_numpy(g[f"{tag}/rep"]), fscale, what="rep")
    mmd = cost.fit_cost(pi)
    w_ref = torch.from_numpy(g[f"{tag}/w"])
    assert_close(cost.w, w_ref, w_ref.abs().max().item(), what="w")
    assert abs(mmd - float(g[f"{tag}/mmd"])) <= 3e-3 * float(g[f"{tag}/mmd"])
    cost.w = w_ref.clone()   # evaluate the costs with the reference's weights: isolates the feature error
    c_ref = torch.from_numpy(g[f"{tag}/costs"])
    cscale = max(c_ref.abs().max().item(), float(w_ref.norm()) * fscale)
    assert_close(cost.get_costs(pi), c_ref, cscale, what="costs")
    assert abs(float(cost.get_expert_cost()) - float(g[f"{tag}/expert_cost"])) <= REL * cscale
    total, info = cost.get_bonus_costs(xs, xa, _FixedDiscEnsemble(torch.from_numpy(g["disc"]), 0.4), next_states=nxt)
    t_ref = torch.from_numpy(g[f"{tag}/total"])
    assert total.shape == t_ref.shape
    assert_close(total, t_ref, t_ref.abs().max().item(), what="total")
    for k in ("bonus", "ipm", "v_targ", "cost"):
        r = torch.from_numpy(g[f"{tag}/info_{k}"])
        assert_close(info[k], r, max(r.abs().max().item(), cscale), what=k)


def test_mlp_cost_default_shape_matches_oracle():
    """The reference's default MLPCost (452 -> 2048 -> 2048 -> 1024) against the fp32 oracle, 1000 rows."""
    from amp_extensions_b200 import MLPCost
    g = torch.Generator().manual_seed(8)
    es = torch.randn(512, 226, generator=g)
    expert = torch.cat([es, es + 0.05 * torch.randn(512, 226, generator=g)], dim=1)
    cost = MLPCost(expert, lambda_b=0.0025, seed=100)
    oc = mo.MlpCostOracle(expert, lambda_b=0.0025, seed=100)
    x = torch.cat([es[:1000 % 512 + 488], es[:1000 % 512 + 488] * 0.9], dim=1)
    x = torch.randn(1000, 452, generator=g)
    rep, rep_ref = cost.get_rep(x), oc.get_rep(x)
    assert_close(rep, rep_ref, (2.0 / 1024) ** 0.5, what="rep")
    assert abs(cost.fit_cost(x) - oc.fit_cost(x)) <= 3e-3 * oc.fit_cost(x)
    cost.w = oc.w.clone()
    c_ref = oc.get_costs(x)
    assert_close(cost.get_costs(x), c_ref, max(c_ref.abs().max().item(), float(oc.w.norm()) * (2.0 / 1024) ** 0.5),
                 what="costs")
    with pytest.raises(Exception):   # a feature-net handle is not an env
        cost.engine().step(torch.zeros(4, 452).cuda(), torch.zeros(4, 0).cuda(), None, None)


@pytest.mark.parametrize("E", [40000, 39999])
def test_full_size_fused_step_properties(E):
    """BASELINE.json configs[1] size through size-independent properties of the fused step (TMA-staged post kernel,
    odd E exercises its trailing unpaired row): s' - s is exactly the active member's delta, the discrepancy equals
    the one computed by the stand-alone entry point (different kernel, different summation order), results are
    equivariant under a permutation of the envs, counters advance by one, the cost is inside its range."""
    from amp_extensions_b200 import RBFLinearCost
    from amp_extensions_b200.engine import HumanoidTermination
    c = H.ns_case()
    eng = make_engine(c, "fp16")
    eng.set_termination(HumanoidTermination(horizon=300))
    cost = RBFLinearCost(H.ns_expert(), feature_dim=512, input_type="ss", bw_quantile=0.1, lambda_b=0.0025, seed=100)
    eng.load_rff(cost.rff.weight.data, cost.rff.bias.data, split=True)
    g = torch.Generator().manual_seed(31)
    s = H.humanoid_like_states(E, seed=33).cuda()
    a = torch.randn(E, 28, generator=g).cuda()
    member = torch.randint(0, 4, (E,), generator=g, dtype=torch.int32).cuda()
    steps = torch.randint(0, 299, (E,), generator=g, dtype=torch.int32).cuda()
    w = (torch.randn(512, generator=g) * 0.02).cuda()
    st = steps.clone()
    nxt, disc, done, cst, ipm, bonus = eng.step_cost(s, a, member, st, w, 0.0025, 0.35)
    assert torch.equal(st, steps + 1)
    # linearity: the same pass's member deltas, re-read through the forward entry point in slices
    for r0 in range(0, E, 8192):
        r1 = min(E, r0 + 8192)
        f = eng.forward(s[r0:r1], a[r0:r1])
        act = f[member[r0:r1].long(), torch.arange(r1 - r0, device="cuda")]
        assert torch.equal(nxt[r0:r1], s[r0:r1] + act)
    d2 = eng.discrepancy(s, a)
    assert_close(disc, d2, d2.mean().item(), rel=2e-6, what="disc (fused vs stand-alone kernel)")
    assert float(cst.min()) >= -1.0 - 1e-6 and float(cst.max()) <= 0.0025 + 1e-6   # (1-l) c - l * bonus, c in [-1, 0]
    assert torch.equal(cst, ipm - bonus)
    perm = torch.randperm(E, generator=g).cuda()
    st2 = steps[perm].clone()
    nxt2, disc2, done2, cst2, _, _ = eng.step_cost(s[perm].contiguous(), a[perm].contiguous(), member[perm].contiguous(),
                                                  st2, w, 0.0025, 0.35)
    assert torch.equal(nxt2, nxt[perm]) and torch.equal(disc2, disc[perm])
    assert torch.equal(done2, done[perm]) and torch.equal(cst2, cst[perm])
    assert 0 < int(done.sum()) < E


# ---------------------------------------------------------------------------------------------------
# GAILCost evaluation side (gail_cost.py:232-283): discriminator through the grouped GEMM, linear head


class _RefDisc:
    """The attributes of the reference Discriminator / GAILCost that the device wrapper reads."""

    def __init__(self, ws, bs, activation="relu"):
        import torch.nn as nn
        lin = [nn.Linear(w.shape[1], w.shape[0]) for w in ws]
        for l, w, b in zip(lin, ws, bs):
            l.weight.data, l.bias.data = w.clone(), b.clone()
        self.activation = nn.ReLU() if activation == "relu" else nn.Tanh()
        if len(lin) == 1:
            self.net = lin[0]
        else:
            layers = [lin[0]]
            for l in lin[1:]:
                layers += [self.activation, l]
            self.net = nn.Sequential(*layers)


class _RefGail:
    def __init__(self, ws, bs, loss_type, lambda_b, input_type="ss"):
        self.disc = _RefDisc(ws, bs)
        self.disc_loss_type, self.lambda_b, self.input_type = loss_type, lambda_b, input_type


@pytest.mark.parametrize("prec", PRECISIONS)
@pytest.mark.parametrize("tag", ["ls_two_hidden", "ll_small", "ls_linear"])
def test_gail_cost_matches_reference(tag, prec):
    import os
    from amp_extensions_b200 import GAILCost
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "gail_golden.npz"))
    n = int(g[f"{tag}/n_linear"])
    ws = [torch.from_numpy(g[f"{tag}/w{i}"]) for i in range(n)]
    bs = [torch.from_numpy(g[f"{tag}/b{i}"]) for i in range(n)]
    ref = _RefGail(ws, bs, str(g[f"{tag}/loss_type"]), float(g[f"{tag}/lambda_b"]))
    cost = GAILCost(ref, precision=prec)
    assert cost.lambda_b == ref.lambda_b                      # attributes are the reference object's
    xs, xa, nxt = (torch.from_numpy(g[k]) for k in ("xs", "xa", "next"))
    ss = torch.cat([xs, nxt], dim=1)
    d_ref = torch.from_numpy(g[f"{tag}/disc_outs"])
    dscale = max(d_ref.abs().max().item(), 1.0)
    assert_close(cost.disc_outputs(ss), d_ref, dscale, what="disc outputs")
    c_ref = torch.from_numpy(g[f"{tag}/costs"])
    # the cost is a smooth function of d with slope <= 0.5 * (1 + |d|): same relative budget on its own scale
    cscale = max(c_ref.abs().max().item(), dscale)
    assert_close(cost.get_costs(ss), c_ref, cscale, what="costs")
    total, info = cost.get_bonus_costs(xs, xa, _FixedDiscEnsemble(torch.from_numpy(g["disc"]), 1.0), next_states=nxt)
    assert_close(total, torch.from_numpy(g[f"{tag}/total"]), cscale, what="total")
    for k in ("bonus", "ipm", "v_targ", "cost"):
        assert_close(info[k], torch.from_numpy(g[f"{tag}/info_{k}"]), cscale, what=k)
    # after an in-place parameter update (what disc_opt.step() does) the packed weights are refreshed
    with torch.no_grad():
        for l in cost._linears():
            l.weight.mul_(0.5)
    ws2 = [w * 0.5 for w in ws]
    d2 = mo.gail_disc_forward(ws2, bs, ss)
    assert_close(cost.disc_outputs(ss), d2, max(d2.abs().max().item(), 1.0), what="disc outputs after update")


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
def test_unaligned_state_rows_take_the_fallback_kernel_with_the_same_results(prec):
    """A state slice that starts on an odd row is only 8-byte aligned: the TMA-staged post kernel needs 16 bytes, so
    the library falls back to the one-warp-per-row kernel.  Same numbers either way (next state and flags bit for
    bit; the discrepancy up to its summation order)."""
    from amp_extensions_b200 import RBFLinearCost
    from amp_extensions_b200.engine import HumanoidTermination
    c = H.ns_case()
    eng = make_engine(c, prec)
    eng.set_termination(HumanoidTermination(horizon=300))
    cost = RBFLinearCost(H.ns_expert(), feature_dim=512, input_type="ss", bw_quantile=0.1, lambda_b=0.0025, seed=100,
                         precision=prec)
    eng.load_rff(cost.rff.weight.data, cost.rff.bias.data, split=True)
    E = 777
    g = torch.Generator().manual_seed(41)
    big = H.humanoid_like_states(E + 1, seed=43).cuda()
    a = torch.randn(E, 28, generator=g).cuda()
    member = torch.randint(0, 4, (E,), generator=g, dtype=torch.int32).cuda()
    w = (torch.randn(512, generator=g) * 0.02).cuda()
    odd = big[1:]                        # data_ptr is 904 bytes past a 256-byte boundary
    assert odd.data_ptr() % 16 == 8 and odd.is_contiguous()
    aligned = odd.clone()
    out_odd = eng.step_cost(odd, a, member, torch.zeros(E, dtype=torch.int32).cuda(), w, 0.0025, 0.35)
    out_al = eng.step_cost(aligned, a, member, torch.zeros(E, dtype=torch.int32).cuda(), w, 0.0025, 0.35)
    assert torch.equal(out_odd[0], out_al[0]) and torch.equal(out_odd[2], out_al[2])
    assert_close(out_odd[1], out_al[1], out_al[1].mean().item(), rel=2e-6, what="disc")
    assert_close(out_odd[3], out_al[3], out_al[3].abs().max().item(), rel=1e-5, what="cost")


def test_column_fused_forward_matches_one_launch_per_layer_bit_for_bit(tmp_path):
    """The default forward pass is ONE launch (csrc/gemm_chain.cuh): a CTA pair runs every layer of a (member, 256-row
    env tile), the activations handed on through L2, the last partial round shared between pairs with the final layer
    as M 256 x N 128 halves.  Every output element accumulates its K blocks in the same order as in the per-layer
    launches (SIMSTEP_CHAIN=0), so ALL outputs of the step are bit-identical - for batches of 1 .. 40 001 rows, i.e.
    with fewer units than CTA pairs, whole rounds only, shared units in the last round (4 800 and 40 001 rows) and a
    plain, unshared last round (7 000 rows: no whole round in sequence, 38 units left over for 74 pairs; 21 500 rows: one
    round in sequence, 40 left over) - and for an irregular second ensemble (three members, no dense connections, tanh,
    hidden 512 / 256 / 512: the pairs sharing a unit get unequal work) at 6 812 and 19 193 rows."""
    import os
    import subprocess
    import sys
    script = os.path.join(os.path.dirname(os.path.abspath(__file__)), "write_step_outputs.py")
    files = {}
    for name in ("per_layer", "default"):
        out = str(tmp_path / f"{name}.npz")
        env = {k: v for k, v in os.environ.items() if k != "SIMSTEP_CHAIN"}
        if name == "per_layer":
            env["SIMSTEP_CHAIN"] = "0"
        res = subprocess.run([sys.executable, script, out], env=env, capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
        files[name] = np.load(out)
    ref, chain = files["per_layer"], files["default"]
    assert sorted(ref.files) == sorted(chain.files)
    for k in ref.files:
        assert np.array_equal(ref[k], chain[k], equal_nan=True), k


def test_column_fused_forward_replays_from_a_cuda_graph_with_shared_units():
    """4 800 rows are 76 units for 74 CTA pairs: two units of the last round are shared between pairs through the
    global tile counters, which the kernel itself leaves clean - so the step can be captured once and replayed (the
    rollout and the single-env plugin do) with bit-identical results, replay after replay."""
    from amp_extensions_b200.engine import Engine, HumanoidTermination
    c = H.ns_case()
    eng = Engine(c["S"], c["A"], c["N"], c["hidden"], dense_connect=True, activation="relu", transform=True,
                 precision="fp16")
    eng.load_ensemble(c["ws"], c["bs"], c["tf"])
    eng.set_termination(HumanoidTermination(enable_velocity_check=True))
    E = 4800
    assert eng.forward_launches(E) == 1
    g = torch.Generator().manual_seed(9)
    s = H.humanoid_like_states(E, seed=3).cuda()
    a = torch.randn(E, 28, generator=g).cuda()
    member = torch.randint(0, 4, (E,), generator=g, dtype=torch.int32).cuda()
    steps0 = torch.zeros(E, dtype=torch.int32, device="cuda")
    ref = eng.step(s, a, member, steps0.clone())
    ref = [t.clone() for t in ref]
    steps = steps0.clone()
    out = [torch.empty_like(t) for t in ref]
    eng.step(s, a, member, steps, next_state=out[0], disc=out[1], done=out[2])      # warm-up outside the capture
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        eng.step(s, a, member, steps, next_state=out[0], disc=out[1], done=out[2])
    for _ in range(3):
        for t in out:
            t.zero_()
        graph.replay()
        torch.cuda.synchronize()
        for got, want in zip(out, ref):
            assert torch.equal(got, want)


def test_workspace_guard_zones_stay_intact(tmp_path):
    """compute-sanitizer is not available on the GPU boxes; SIMSTEP_DEBUG_GUARDS=1 puts every workspace buffer between
    two 64 KB guard zones instead (simstep_debug_check_guards).  A separate process (the switch is read at
    simstep_create) runs the step + cost at ragged and tile-aligned batch sizes - one launch per layer, the
    column-fused forward kernel with whole rounds only, with shared units, and the chunked path - and no guard byte
    may change."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = r'''
import sys, torch
sys.path.insert(0, %r)
from oracle import milo_oracle as mo
from tests import helpers as H
from amp_extensions_b200.engine import Engine, HumanoidTermination
c = H.ns_case()
for prec, chunk in (("fp16", 0), ("tf32", 0), ("fp16", 4096)):
    eng = Engine(c["S"], c["A"], c["N"], c["hidden"], dense_connect=True, activation="relu", transform=True,
                 precision=prec, **({"max_chunk_envs": chunk} if chunk else {}))
    eng.load_ensemble(c["ws"], c["bs"], c["tf"])
    eng.set_termination(HumanoidTermination(enable_velocity_check=True))
    oc = mo.RffCostOracle(H.ns_expert(), feature_dim=512, input_type="ss", bw_quantile=0.1, lambda_b=0.0025, seed=100)
    eng.load_rff(oc.rff_weight, oc.rff_bias, split=True)
    g = torch.Generator().manual_seed(1)
    w = (torch.randn(512, generator=g) * 0.01).cuda()
    for E in (1, 255, 256, 257, 4800, 9473, 20001):
        s = H.humanoid_like_states(E, seed=E %% 5).cuda()
        a = torch.randn(E, 28, generator=g).cuda()
        member = torch.randint(0, 4, (E,), generator=g, dtype=torch.int32).cuda()
        steps = torch.zeros(E, dtype=torch.int32, device="cuda")
        for split in (True, False):
            eng.set_rff_split(split)
            eng.step_cost(s, a, member, steps, w, 0.0025, c["threshold"])
        eng.discrepancy(s, a)
    n, bad = eng.check_guards()
    print("GUARDS", prec, chunk, n, bad)
    assert n >= 4 and bad == 0, (prec, chunk, n, bad)
''' % root
    for chain in ("0", "2"):
        env = dict(os.environ, SIMSTEP_DEBUG_GUARDS="1", SIMSTEP_CHAIN=chain)
        res = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
        assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-3000:]
        assert res.stdout.count("GUARDS") == 3
