"""GPU parity of the rollout helpers (SURVEY.md section 8f ranks 1-2) through the C ABI: Gaussian MLP policy,
discounted sums / GAE, auto-reset and the whole DeviceRollout loop against the oracle.

Tolerances: the policy network and the discounted sums are plain fp32 on the CUDA cores; they differ from the
reference's fp32 only by summation order (<= 2e-6 relative to the output scale, written below).  The rollout loop
inherits the env step's 1e-3 budget (BASELINE.json north_star) per step.
"""
import os

import numpy as np
import pytest
import torch

from oracle import milo_oracle as mo
from oracle import rollout_oracle as ro
from tests import helpers as H
from tests.test_parity_gpu import assert_close, make_engine

pytestmark = pytest.mark.gpu

G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "rollout_golden.npz"))


class _FC:
    def __init__(self, ws, bs, nonlinearity, in_shift=None, in_scale=None, out_shift=None, out_scale=None):
        self.fc_layers = [torch.nn.Linear(w.shape[1], w.shape[0]) for w in ws]
        for l, w, b in zip(self.fc_layers, ws, bs):
            l.weight.data, l.bias.data = w.clone(), b.clone()
        self.nonlinearity = torch.relu if nonlinearity == "relu" else torch.tanh
        obs, act = ws[0].shape[1], ws[-1].shape[0]
        self.in_shift = torch.zeros(obs) if in_shift is None else torch.as_tensor(in_shift)
        self.in_scale = torch.ones(obs) if in_scale is None else torch.as_tensor(in_scale)
        self.out_shift = torch.zeros(act) if out_shift is None else torch.as_tensor(out_shift)
        self.out_scale = torch.ones(act) if out_scale is None else torch.as_tensor(out_scale)


class _Policy:
    """The attributes of mjrl's MLP policy that DeviceRollout reads (gaussian_mlp.py:36-44)."""

    def __init__(self, model, log_std):
        self.model, self.log_std = model, torch.as_tensor(log_std)


def _golden_policy(tag, n_layers):
    ws = [torch.from_numpy(G[f"{tag}/w{i}"]) for i in range(n_layers)]
    bs = [torch.from_numpy(G[f"{tag}/b{i}"]) for i in range(n_layers)]
    return ws, bs


def _tiny_engine():
    c = H.tiny_case("tiny_dense")
    return c, make_engine(c, "fp16")


def test_policy_mean_matches_reference_default_transformations():
    _, eng = _tiny_engine()
    ws, bs = _golden_policy("polA", 3)
    eng.load_policy(ws, bs, "tanh", log_std=G["polA/log_std"])
    obs = torch.from_numpy(G["polA/obs"]).cuda()
    action, mean = eng.policy_act(obs)
    ref = torch.from_numpy(G["polA/mean"])
    assert_close(mean, ref, ref.abs().max().item(), rel=2e-6, what="policy mean")
    assert torch.equal(action, mean)  # no noise: the evaluation action
    # get_action with the reference's own numpy draws (float64 there, fp32 here)
    noise = torch.from_numpy(G["polA/noise"]).float().cuda()
    act8, _ = eng.policy_act(obs[:8].contiguous(), noise)
    ref8 = torch.from_numpy(G["polA/get_action"])
    assert_close(act8, ref8, ref8.abs().max().item(), rel=2e-6, what="get_action")


def test_policy_relu_with_transformations_and_ragged_batches():
    _, eng = _tiny_engine()
    ws, bs = _golden_policy("polB", 4)
    eng.load_policy(ws, bs, "relu", G["polB/in_shift"], G["polB/in_scale"], G["polB/out_shift"], G["polB/out_scale"])
    ref = torch.from_numpy(G["polB/mean"])
    for n in (50, 1, 3, 17):  # group size is 4 envs per warp: ragged tails
        obs = torch.from_numpy(G["polB/obs"][:n]).cuda().contiguous()
        _, mean = eng.policy_act(obs)
        assert_close(mean, ref[:n], ref.abs().max().item(), rel=2e-6, what=f"policy mean n={n}")
    # empty batch is a no-op
    eng.policy_act(torch.empty((0, 40), device="cuda"))


def test_policy_requires_load_and_validates_sizes():
    from amp_extensions_b200 import _lib
    _, eng = _tiny_engine()
    with pytest.raises(_lib.SimstepError):
        eng.policy_obs_dim, eng.policy_act_dim = 4, 2
        eng.policy_act(torch.zeros((4, 4), device="cuda"))
    with pytest.raises(_lib.SimstepError):  # layer sizes do not chain
        eng.load_policy([torch.zeros(8, 4), torch.zeros(2, 9)], [torch.zeros(8), torch.zeros(2)])
    with pytest.raises(_lib.SimstepError):  # too wide
        eng.load_policy([torch.zeros(4096, 4)], [torch.zeros(4096)])


def test_discount_matches_process_samples_golden():
    """Ragged trajectories, one per env column, exactly the reference's paths (float64 there, fp32 here)."""
    _, eng = _tiny_engine()
    gamma, lam = [float(x) for x in G["ps/gamma_lambda"]]
    lens, term = G["ps/lens"], G["ps/terminated"]
    T, E = int(lens.max()), len(lens)
    rew, base = np.zeros((T, E), np.float32), np.zeros((T, E), np.float32)
    for i, n in enumerate(lens):
        rew[:n, i], base[:n, i] = G[f"ps/rewards{i}"], G[f"ps/baseline{i}"]
    ret, adv = eng.discount(torch.from_numpy(rew).cuda(), gamma, baseline=torch.from_numpy(base).cuda(),
                            gae_lambda=lam, lengths=torch.from_numpy(lens.astype(np.int32)).cuda(),
                            terminated=torch.from_numpy(term.astype(np.uint8)).cuda())
    for i, n in enumerate(lens):
        r_ref, a_ref = torch.from_numpy(G[f"ps/returns{i}"]), torch.from_numpy(G[f"ps/advantages{i}"])
        assert_close(ret[:n, i], r_ref, r_ref.abs().max().item(), rel=1e-5, what=f"returns path {i}")
        assert_close(adv[:n, i], a_ref, a_ref.abs().max().item(), rel=1e-5, what=f"advantages path {i}")
        assert not ret[n:, i].any() and not adv[n:, i].any()


def test_discount_segments_within_a_column():
    """Several trajectories back to back in one env column, cut at seg_end flags."""
    _, eng = _tiny_engine()
    rng = np.random.default_rng(0)
    T, E, gamma, lam = 97, 33, 0.99, 0.95
    rew, base = rng.normal(size=(T, E)).astype(np.float32), rng.normal(size=(T, E)).astype(np.float32)
    seg = (rng.random((T, E)) < 0.08).astype(np.uint8)
    seg[:, 0] = 0
    seg[:, 1] = 1  # every step is its own terminated trajectory
    term = seg[T - 1].copy()
    ret, adv = eng.discount(torch.from_numpy(rew).cuda(), gamma, baseline=torch.from_numpy(base).cuda(), gae_lambda=lam,
                            seg_end=torch.from_numpy(seg).cuda(), terminated=torch.from_numpy(term).cuda())
    ret, adv = ret.cpu().numpy(), adv.cpu().numpy()
    for e in range(E):
        t0 = 0
        ends = list(np.flatnonzero(seg[:, e]))
        if not ends or ends[-1] != T - 1:
            ends.append(T - 1)
        for t1 in ends:
            terminated = bool(seg[t1, e])
            r_ref = ro.discount_sum(rew[t0:t1 + 1, e].astype(np.float64), gamma)
            a_ref = ro.gae_advantages(rew[t0:t1 + 1, e].astype(np.float64), base[t0:t1 + 1, e].astype(np.float64),
                                      terminated, gamma, lam)
            np.testing.assert_allclose(ret[t0:t1 + 1, e], r_ref, rtol=0, atol=2e-5 * max(1.0, np.abs(r_ref).max()))
            np.testing.assert_allclose(adv[t0:t1 + 1, e], a_ref, rtol=0, atol=2e-5 * max(1.0, np.abs(a_ref).max()))
            t0 = t1 + 1


def test_auto_reset_is_exact():
    c, eng = _tiny_engine()
    E, S, N = 1000, c["S"], c["N"]
    g = torch.Generator(device="cuda").manual_seed(3)
    nxt = torch.randn(E, S, device="cuda", generator=g)
    pool = torch.randn(37, S, device="cuda", generator=g)
    done = (torch.rand(E, device="cuda", generator=g) < 0.4).to(torch.uint8)
    pick = torch.randint(0, 1000, (E,), device="cuda", generator=g, dtype=torch.int32)
    member = torch.randint(0, N, (E,), device="cuda", generator=g, dtype=torch.int32)
    steps = torch.randint(0, 300, (E,), device="cuda", generator=g, dtype=torch.int32)
    m0, s0 = member.clone(), steps.clone()
    out = torch.full((E, S), float("nan"), device="cuda")
    eng.auto_reset(nxt, done, pool, pick, out, member, steps)
    d = done.bool()
    assert torch.equal(out, torch.where(d[:, None], pool[(pick % 37).long()], nxt))
    assert torch.equal(member, torch.where(d, (m0 + 1) % N, m0))
    assert torch.equal(steps, torch.where(d, torch.zeros_like(s0), s0))


@pytest.mark.parametrize("with_cost", [False, True])
def test_device_rollout_matches_oracle_loop(with_cost):
    """The whole loop (policy -> step -> cost -> auto-reset) against the oracle's batched restatement of the sampler,
    same noise and reset picks on both sides.  Errors compound over steps through the learned dynamics, so the
    per-step 1e-3 budget is checked on a short horizon; termination flags must agree except inside the band."""
    from amp_extensions_b200 import AmpDataset, DynamicsEnsemble, RBFLinearCost, VecSimEnv
    from amp_extensions_b200.rollout import DeviceRollout
    c = H.ns_case()
    S, A, N, E, T, horizon = 226, 28, 4, 96, 6, 4
    s, a, s2 = H.synth_dataset(2048, S, A, 0)
    ds = AmpDataset(s, a, s2)
    ens = DynamicsEnsemble(S, A, ds, None, num_models=N, hidden_sizes=c["hidden"], dense_connect=True, transform=True,
                           base_seed=100)
    ens.threshold = 0.4
    pool = H.humanoid_like_states(64, 5, fall_fraction=0.0)
    pool[:, 0] = 1.5  # start well above the ground: falls happen through the dynamics, not at reset
    env = VecSimEnv(ens, E, horizon=horizon, reset_states=pool, seed=1)
    env.reset(initial_states=pool[torch.arange(E) % 64])
    cost_o = None
    if with_cost:
        expert = H.ns_expert()
        cost = RBFLinearCost(expert, feature_dim=512, input_type="ss", bw_quantile=0.1, lambda_b=0.0025, seed=100)
        cost.fit_cost(torch.cat([s[:256], s2[:256]], dim=1))
        env.attach_cost(cost)
        cost_o = mo.RffCostOracle(expert, feature_dim=512, input_type="ss", bw_quantile=0.1, lambda_b=0.0025, seed=100)
        cost_o.w = cost.w
    ws, bs = _golden_policy("polA", 3)
    pol = _Policy(_FC(ws, bs, "tanh"), G["polA/log_std"])
    ro_dev = DeviceRollout(env, pol, seed=0)
    g = torch.Generator().manual_seed(9)
    noise = torch.randn(T, E, A, generator=g)
    pick = torch.randint(0, 64, (T, E), generator=g, dtype=torch.int32)
    member0, steps0, ob0 = env.member.cpu().numpy(), env.num_steps.cpu().numpy(), env.ob.cpu().numpy()
    batch = ro_dev.collect(T, noise=noise.cuda(), pick=pick.cuda())
    wsE = [[l.weight.data for l in m.model.fc_layers] for m in ens.models]
    bsE = [[l.bias.data for l in m.model.fc_layers] for m in ens.models]
    ref = ro.rollout(wsE, bsE, ens.transformations, dict(ws=ws, bs=bs, log_std=G["polA/log_std"]), ob0, member0, steps0,
                     pool.numpy(), noise.numpy(), pick.numpy(), horizon=horizon, cost=cost_o, threshold=ens.threshold,
                     n_models=N)
    done_dev, done_ref = batch.done.cpu().numpy().astype(bool), ref["done"]
    # every env hits the horizon at least once in T > horizon steps, so auto-reset is exercised
    assert done_ref.any() and (~done_ref).any()
    agree = done_dev == done_ref
    assert agree.mean() > 0.99
    # compare every step up to (and including) an env's first disagreement-free prefix
    ok = np.logical_and.accumulate(agree, axis=0)
    ok = np.concatenate([np.ones((1, E), bool), ok[:-1]], axis=0)  # step t is comparable if flags agreed before t
    m = torch.from_numpy(ok)
    for name, scale in (("observations", 1.0), ("next_observations", 1.0), ("actions", 1.0), ("means", 0.1)):
        x, r = getattr(batch, name).cpu(), torch.from_numpy(ref[name])
        assert_close(x[m], r[m], scale, rel=3e-3, what=name)  # T compounding steps of a 1e-3-per-step budget
    assert_close(batch.disc.cpu()[m], torch.from_numpy(ref["disc"])[m], float(ref["disc"].mean()), rel=3e-3, what="disc")
    if with_cost:
        assert_close(batch.cost.cpu()[m], torch.from_numpy(ref["cost"])[m], float(np.abs(ref["cost"]).max()), rel=3e-3,
                     what="cost")
        assert torch.equal(batch.rewards, -batch.cost)
    # path layout (sampler.py:70-81)
    paths = batch.paths()
    assert sum(len(p["rewards"]) for p in paths) == T * E
    p0 = paths[0]
    assert p0["observations"].dtype == np.float64 and p0["observations"].shape[1] == S
    assert set(p0["agent_infos"]) == {"mean", "log_std", "evaluation"} and p0["env_infos"][0]["valid"]
    assert all(p["terminated"] for p in batch.paths(include_partial=False))
    for p in paths:  # within a trajectory the next observation is the following observation
        assert np.array_equal(p["observations"][1:], p["next_observations"][:-1])
    # returns over the segmented columns equal per-path discount sums
    ret = batch.returns(0.99).cpu().numpy()
    for (e, t0, t1, _), p in zip(batch.segments(), paths):
        np.testing.assert_allclose(ret[t0:t1, e], ro.discount_sum(p["rewards"], 0.99), rtol=0, atol=1e-5)
    st = batch.statistics()
    assert len(st["ep_len"]) == len(paths) and sum(st["ep_len"]) == T * E


def test_sample_paths_contract():
    """sample_points's contract (sampler.py:30-34): at least num_to_collect samples, complete trajectories only."""
    from amp_extensions_b200 import AmpDataset, DynamicsEnsemble, VecSimEnv
    from amp_extensions_b200.rollout import DeviceRollout
    c = H.tiny_case("tiny_dense")
    S, A = c["S"], c["A"]
    s, a, s2 = c["ds"]
    ens = DynamicsEnsemble(S, A, AmpDataset(s, a, s2), None, num_models=c["N"], hidden_sizes=c["hidden"],
                           dense_connect=True, transform=True, base_seed=100)
    from amp_extensions_b200 import HumanoidTermination
    term = HumanoidTermination(horizon=7, fall_contact_bodies=())
    env = VecSimEnv(ens, 16, termination=term, reset_states=s[:32], seed=0)
    g = torch.Generator().manual_seed(0)
    ws = [torch.randn(8, S, generator=g) * 0.1, torch.randn(A, 8, generator=g) * 0.1]
    bs = [torch.zeros(8), torch.zeros(A)]
    ro_dev = DeviceRollout(env, _Policy(_FC(ws, bs, "tanh"), np.full(A, -1.0, np.float32)), seed=0)
    paths, n = ro_dev.sample_paths(300, mode="samples")
    assert n >= 300 and n == sum(len(p["rewards"]) for p in paths)
    assert all(p["terminated"] and len(p["rewards"]) == 7 for p in paths)  # horizon-only termination
    paths, _ = ro_dev.sample_paths(20, mode="trajectories", eval_mode=True)
    assert len(paths) >= 20
    assert all(np.array_equal(p["actions"], p["agent_infos"]["mean"].astype(np.float64)) for p in paths)


def test_graph_replay_equals_eager_loop():
    """collect(graph=True) replays the same launches from a CUDA graph: bit-identical buffers, and the env's
    counters advance exactly as in the eager loop (also on a second replay of the cached graph)."""
    from amp_extensions_b200 import AmpDataset, DynamicsEnsemble, HumanoidTermination, VecSimEnv
    from amp_extensions_b200.rollout import DeviceRollout
    c = H.tiny_case("tiny_dense")
    S, A = c["S"], c["A"]
    s, a, s2 = c["ds"]
    ens = DynamicsEnsemble(S, A, AmpDataset(s, a, s2), None, num_models=c["N"], hidden_sizes=c["hidden"],
                           dense_connect=True, transform=True, base_seed=100)
    g = torch.Generator().manual_seed(0)
    ws = [torch.randn(8, S, generator=g) * 0.1, torch.randn(A, 8, generator=g) * 0.1]
    bs = [torch.zeros(8), torch.zeros(A)]
    pol = _Policy(_FC(ws, bs, "tanh"), np.full(A, -1.0, np.float32))
    T, E = 9, 50
    noise = torch.randn(2, T, E, A, generator=g).cuda()
    pick = torch.randint(0, 32, (2, T, E), generator=g, dtype=torch.int32).cuda()
    outs = []
    for use_graph in (False, True):
        env = VecSimEnv(ens, E, termination=HumanoidTermination(horizon=4, fall_contact_bodies=()),
                        reset_states=s[:32], seed=0)
        env.reset(initial_states=s[:E])
        ro_dev = DeviceRollout(env, pol, seed=0)
        got = []
        for k in range(2):
            b = ro_dev.collect(T, noise=noise[k], pick=pick[k], graph=use_graph)
            got.append({n: getattr(b, n).clone() for n in ("observations", "next_observations", "actions", "disc",
                                                            "done")})
            got[-1].update(member=env.member.clone(), num_steps=env.num_steps.clone(), ob=env.ob.clone())
        outs.append(got)
    for k in range(2):
        for n, v in outs[0][k].items():
            assert torch.equal(v, outs[1][k][n]), (k, n)


def test_graph_replay_survives_policy_and_cost_reloads():
    """ADVICE r1: load_policy() frees and re-allocates the packed policy, attach_cost() / set_cost_weights() the rff
    buffers and weights - a graph captured before must not be replayed afterwards.  The cache key carries the engine's
    parameter generation and holds one entry: collect(graph=True) after a reload equals the eager loop with the NEW
    parameters, and the cache does not grow."""
    from amp_extensions_b200 import (AmpDataset, DynamicsEnsemble, HumanoidTermination, RBFLinearCost, VecSimEnv)
    from amp_extensions_b200.rollout import DeviceRollout
    c = H.tiny_case("tiny_dense")
    S, A = c["S"], c["A"]
    s, a, s2 = c["ds"]
    ens = DynamicsEnsemble(S, A, AmpDataset(s, a, s2), None, num_models=c["N"], hidden_sizes=c["hidden"],
                           dense_connect=True, transform=True, base_seed=100)
    ens.threshold = 0.5
    cost = RBFLinearCost(torch.cat([s[:64], s2[:64]], dim=1), feature_dim=64, input_type="ss", bw_quantile=0.1,
                         lambda_b=0.1, seed=3)
    cost.fit_cost(torch.cat([s[64:128], s2[64:128]], dim=1))
    g = torch.Generator().manual_seed(0)

    def policy(scale):
        ws = [torch.randn(8, S, generator=g) * scale, torch.randn(A, 8, generator=g) * scale]
        return _Policy(_FC(ws, [torch.zeros(8), torch.zeros(A)], "tanh"), np.full(A, -1.0, np.float32))

    T, E = 5, 40
    noise = torch.randn(3, T, E, A, generator=g).cuda()
    pick = torch.randint(0, 32, (3, T, E), generator=g, dtype=torch.int32).cuda()
    pols = [policy(0.1), policy(0.3), policy(0.2)]
    ws_cost = [cost.w.clone(), cost.w * -2.0, cost.w * 0.5]
    outs = []
    for use_graph in (False, True):
        env = VecSimEnv(ens, E, termination=HumanoidTermination(horizon=4, fall_contact_bodies=()),
                        reset_states=s[:32], seed=0, cost=cost)
        env.reset(initial_states=s[:E])
        ro_dev = DeviceRollout(env, pols[0], seed=0)
        got = []
        for k in range(3):
            ro_dev.load_policy(pols[k])            # re-allocates the packed policy on the device
            if k == 1:
                env.attach_cost(cost)              # re-allocates the rff buffers
            env.set_cost_weights(ws_cost[k])       # in place after the first call
            b = ro_dev.collect(T, noise=noise[k], pick=pick[k], graph=use_graph)
            got.append({n: getattr(b, n).clone() for n in ("observations", "actions", "cost", "done")})
            if use_graph:
                assert len(ro_dev._graphs) == 1
        outs.append(got)
    for k in range(3):
        for n, v in outs[0][k].items():
            assert torch.equal(v, outs[1][k][n]), (k, n)
    assert not torch.equal(outs[1][0]["actions"], outs[1][1]["actions"])  # the reloads did change the results


def test_moments_and_whitening_match_numpy():
    """compute_advantages(normalize=True) (process_samples.py:14-19): numpy float64 mean / population std."""
    _, eng = _tiny_engine()
    rng = np.random.default_rng(5)
    for n in (1, 7, 1000, 300 * 4001):
        x = (rng.normal(size=n) * 3 + 0.7).astype(np.float32)
        valid = (rng.random(n) < 0.8).astype(np.uint8)
        valid[0] = 1
        xd, vd = torch.from_numpy(x).cuda(), torch.from_numpy(valid).cuda()
        for v_np, v_dev in ((None, None), (valid, vd)):
            sel = x.astype(np.float64) if v_np is None else x.astype(np.float64)[v_np.astype(bool)]
            st = eng.moments(xd, v_dev).cpu().numpy()
            assert st[0] == sel.size
            assert abs(st[1] - sel.sum()) <= 1e-9 * max(1.0, np.abs(sel).sum())
            assert abs(st[2] - (sel ** 2).sum()) <= 1e-9 * (sel ** 2).sum()
            out = eng.whiten(xd, torch.from_numpy(st).cuda(), v_dev).cpu().numpy()
            ref = (x.astype(np.float64) - sel.mean()) / (sel.std() + 1e-8)
            if v_np is not None:
                ref = np.where(v_np.astype(bool), ref, 0.0)
            if sel.size > 1:
                np.testing.assert_allclose(out, ref, rtol=0, atol=2e-6 * max(1.0, np.abs(ref).max()))
    # empty input: count 0, nothing written
    st = eng.moments(torch.empty(0, device="cuda")).cpu().numpy()
    assert st.tolist() == [0.0, 0.0, 0.0]


def test_histogram_kernel_and_device_quantile_match_torch():
    """simstep_histogram against torch.histc-style counting in fp64, and parallel.global_quantile's device path against
    torch.quantile (single process: the all-reduces are identities; tests/test_quantile.py covers adversarial data)."""
    from amp_extensions_b200 import parallel
    _, eng = _tiny_engine()
    g = torch.Generator(device="cuda").manual_seed(2)
    x = torch.rand(200_003, device="cuda", generator=g) ** 3 * 0.7
    lo, hi, bins = 0.05, 0.6, 4096
    counts = eng.histogram(x, lo, hi, bins).cpu()
    xd = x.double().cpu()
    sel = (xd >= lo) & (xd <= hi)
    idx = torch.clamp(((xd[sel] - lo) / ((hi - lo) / bins)).floor(), 0, bins - 1).long()
    assert torch.equal(counts, torch.bincount(idx, minlength=bins))
    assert int(eng.histogram(torch.empty(0, device="cuda"), 0.0, 1.0, 16).sum()) == 0
    for q in (0.1, 0.5, 0.9, 0.999):
        got = parallel.global_quantile(x, q, engine=eng)
        ref = float(torch.quantile(xd, q))
        assert abs(got - ref) <= 1e-6 * float(xd.max() - xd.min()), (q, got, ref)


def test_device_rollout_matches_the_reference_sampler():
    """tests/golden/sampler_golden.npz: the reference's own get_samples + SimEnv + DynamicsEnsemble + MLP policy, six
    trajectories.  Here each trajectory is one env column of DeviceRollout.collect, started from the same state and
    member, fed the same exploration draws; the prefix up to the reference trajectory's end must agree (1e-3 per
    step of the state scale 1.0), and the column must signal `done` at the same step unless the deciding height is
    within 1e-3 of its threshold."""
    from amp_extensions_b200 import AmpDataset, DynamicsEnsemble, VecSimEnv
    from amp_extensions_b200.rollout import DeviceRollout
    from tests.test_parity_gpu import collision_margin
    from tests.test_rollout_oracle import sampler_golden, sampler_noise
    g = sampler_golden()
    S, A = 226, 28
    N, hidden, horizon = int(g["N"]), [int(h) for h in g["hidden"]], int(g["horizon"])
    ds = AmpDataset(*H.synth_dataset(int(g["dataset_rows"]), S, A, int(g["dataset_seed"])))
    ens = DynamicsEnsemble(S, A, ds, None, num_models=N, hidden_sizes=hidden, dense_connect=True, transform=True,
                           base_seed=int(g["base_seed"]))
    got = [[float(l.weight.data.double().abs().sum()) for l in m.model.fc_layers] for m in ens.models]
    np.testing.assert_allclose(got, g["weight_checksum"], rtol=1e-12)
    n_traj, T, _ = g["actions"].shape
    ob0 = torch.from_numpy(g["observations"][:, 0]).float()
    env = VecSimEnv(ens, n_traj, horizon=horizon, reset_states=ob0, seed=1)
    env.reset(initial_states=ob0)
    env.member.copy_(torch.from_numpy(g["member"]).to(torch.int32))
    ws = [torch.from_numpy(g[f"pol_w{i}"]) for i in range(3)]
    bs = [torch.from_numpy(g[f"pol_b{i}"]) for i in range(3)]
    pol = _Policy(_FC(ws, bs, "tanh"), g["log_std"])
    noise = torch.from_numpy(sampler_noise(g)).float().cuda()
    batch = DeviceRollout(env, pol, seed=0).collect(T, noise=noise, pick=torch.zeros((T, n_traj), dtype=torch.int32).cuda())
    done = batch.done.cpu().numpy().astype(bool)
    for k in range(n_traj):
        n = int(g["length"][k])
        for name in ("observations", "next_observations", "actions", "means"):
            x = getattr(batch, name).cpu().numpy()[:n, k]
            err = np.abs(x - g[name][k, :n]).max(axis=1)
            assert (err < 1e-3 * np.arange(1, n + 1)).all(), (k, name, err)
        first = int(np.argmax(done[:, k])) + 1 if done[:, k].any() else None
        if first != n:
            t = min(n, first or n) - 1
            assert collision_margin(g["next_observations"][k, t][None])[0] < 1e-3, (k, first, n)


def test_sampler_shim_matches_the_reference_sampler_on_gpu():
    """amp_extensions_b200.sampler.get_samples (the drop-in for milo/milo/sampler.py) with its default device backend:
    the reference's own get_samples run (tests/golden/sampler_golden.npz) reproduced through SimEnv + DeviceRollout,
    same seeds, same numpy draws, to 1e-3 per step; lengths equal unless the deciding height is within 1e-3 of its
    threshold.  (tests/test_sampler_shim.py checks the host logic exactly, on the CPU oracle.)"""
    from amp_extensions_b200 import AmpDataset, DynamicsEnsemble, SimEnv, sampler
    from tests.test_parity_gpu import collision_margin
    from tests.test_rollout_oracle import sampler_golden
    g = sampler_golden()
    S, A = 226, 28
    N, hidden, horizon = int(g["N"]), [int(h) for h in g["hidden"]], int(g["horizon"])
    ds = AmpDataset(*H.synth_dataset(int(g["dataset_rows"]), S, A, int(g["dataset_seed"])))
    ens = DynamicsEnsemble(S, A, ds, None, num_models=N, hidden_sizes=hidden, dense_connect=True, transform=True,
                           base_seed=int(g["base_seed"]))
    calls = []

    def reset_fn(n, rng):   # the reference drew these from its simulator; trajectory k starts where the golden one did
        calls.append(1)
        return g["observations"][len(calls) - 1, 0][None]

    env = SimEnv(ens, horizon=horizon, reset_fn=reset_fn, seed=1)
    ws = [torch.from_numpy(g[f"pol_w{i}"]) for i in range(3)]
    bs = [torch.from_numpy(g[f"pol_b{i}"]) for i in range(3)]
    pol = _Policy(_FC(ws, bs, "tanh"), g["log_std"])
    n_traj = g["actions"].shape[0]
    paths, n = sampler.get_samples(env, pol, n_traj, int(g["seed"]), mode="trajectories")
    assert len(paths) == n_traj and n == sum(len(p["rewards"]) for p in paths)
    for k, p in enumerate(paths):
        n_ref, n_got = int(g["length"][k]), len(p["rewards"])
        m = min(n_ref, n_got)
        for name, ref in (("observations", g["observations"]), ("next_observations", g["next_observations"]),
                          ("actions", g["actions"])):
            err = np.abs(p[name][:m] - ref[k, :m]).max(axis=1)
            assert (err < 1e-3 * np.arange(1, m + 1)).all(), (k, name, err)
        if n_ref != n_got:
            assert collision_margin(g["next_observations"][k, m - 1][None])[0] < 1e-3, (k, n_got, n_ref)


def test_reward_replacement_matches_the_reference_train_step():
    """The drop-in claim of SURVEY.md section 8(b) on the reference's own numbers: BatchREINFORCE.train_step's reward
    replacement (batch_reinforce.py:103-169) — the lines in tests.helpers.reward_replacement — run over THIS package's
    RBFLinearCost and DynamicsEnsemble must give what the reference's train_step gave over the reference classes
    (tests/golden/trainstep_golden.npz): threshold, fitted w, mb_mmd, bonus_mmd, per-trajectory int / ext sums and
    every replaced reward, to 1e-3 of each quantity's scale."""
    from amp_extensions_b200 import AmpDataset, DynamicsEnsemble, RBFLinearCost
    g = H.trainstep_golden()
    S, A = 226, 28
    N, hidden = int(g["N"]), [int(h) for h in g["hidden"]]
    ds = AmpDataset(*H.synth_dataset(int(g["dataset_rows"]), S, A, int(g["dataset_seed"])))
    ens = DynamicsEnsemble(S, A, ds, None, num_models=N, hidden_sizes=hidden, dense_connect=True, transform=True,
                           base_seed=int(g["base_seed"]))
    ens.compute_threshold()
    assert abs(ens.threshold - float(g["threshold"])) < 1e-3 * float(g["threshold"])
    cost = RBFLinearCost(torch.from_numpy(g["expert"]), feature_dim=int(g["feature_dim"]), input_type="ss",
                         bw_quantile=float(g["bw_quantile"]), lambda_b=float(g["lambda_b"]), seed=int(g["cost_seed"]))
    assert abs(cost.bw - float(g["cost_bw"])) < 1e-6 * float(g["cost_bw"])
    paths = H.trainstep_paths(g)
    infos = H.reward_replacement(paths, cost, ens)
    w_scale = float(np.abs(g["cost_w"]).max())
    assert float(np.abs(cost.w.cpu().numpy() - g["cost_w"]).max()) < 1e-3 * w_scale
    assert abs(float(infos["mb_mmd"]) - float(g["mb_mmd"])) < 1e-3 * float(g["mb_mmd"])
    r_scale = float(np.abs(g["rewards"]).max())
    for k, p in enumerate(paths):
        n = len(p["rewards"])
        assert p["rewards"].shape == (n,)
        assert float(np.abs(p["rewards"] - g["rewards"][k, :n]).max()) < 1e-3 * r_scale, k
    assert infos["ep_len"] == list(g["info_ep_len"])
    for key in ("int", "ext", "reward"):
        ref = g[f"info_{key}"]
        assert float(np.abs(np.asarray(infos[key]) - ref).max()) < 1e-3 * max(float(np.abs(ref).max()), r_scale), key
    assert abs(infos["bonus_mmd"] - float(g["bonus_mmd"])) < 1e-3 * max(abs(float(g["bonus_mmd"])), r_scale)


def test_host_path_stream_downloads_behind_the_next_collect():
    """HostPathStream: batch k is copied to pinned memory on a copy stream while collect() k+1 is already queued; what
    arrives equals a plain .cpu() of the same batch, batches come back in submission order, and a third submit without
    a collect is refused."""
    from amp_extensions_b200 import AmpDataset, DynamicsEnsemble, HumanoidTermination, VecSimEnv
    from amp_extensions_b200.rollout import DeviceRollout, HostPathStream
    c = H.tiny_case("tiny_dense")
    S, A = c["S"], c["A"]
    s, a, s2 = c["ds"]
    ens = DynamicsEnsemble(S, A, AmpDataset(s, a, s2), None, num_models=c["N"], hidden_sizes=c["hidden"],
                           dense_connect=True, transform=True, base_seed=100)
    env = VecSimEnv(ens, 48, termination=HumanoidTermination(horizon=5, fall_contact_bodies=()), reset_states=s[:32],
                    seed=0)
    env.reset()
    g = torch.Generator().manual_seed(0)
    ws = [torch.randn(8, S, generator=g) * 0.1, torch.randn(A, 8, generator=g) * 0.1]
    bs = [torch.zeros(8), torch.zeros(A)]
    ro = DeviceRollout(env, _Policy(_FC(ws, bs, "tanh"), np.full(A, -1.0, np.float32)), seed=0)
    dl = HostPathStream(env.device)
    b0 = ro.collect(6)
    dl.submit(b0)
    b1 = ro.collect(6)
    dl.submit(b1)
    with pytest.raises(RuntimeError):
        dl.submit(b1)
    for b in (b0, b1):
        host = dl.collect()
        for n in HostPathStream.NAMES:
            assert torch.equal(host[n], getattr(b, n).cpu()), n
    assert dl.bytes_per_batch == sum(getattr(b1, n).numel() * getattr(b1, n).element_size() for n in HostPathStream.NAMES)
    with pytest.raises(RuntimeError):
        dl.collect()
