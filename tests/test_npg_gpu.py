"""GPU tests of the on-device NPG step (csrc/npg.cuh through amp_extensions_b200.npg) against the float64 oracle
(oracle/npg_oracle.py), on the same rows.  The kernels are fp32 FMAs summed per CTA, then fp64 across CTAs: the gradient
and Fisher-vector sums are checked to 1e-4 relative L2 at small n and 1e-3 at 1.28 M rows; a whole update to 1e-3."""
import os

import numpy as np
import pytest
import torch

from oracle import npg_oracle as no
from tests import helpers as H
from tests.test_parity_gpu import make_engine

pytestmark = pytest.mark.gpu

G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "rollout_golden.npz"))


def _engine():
    return make_engine(H.tiny_case("tiny_dense"), "fp16")


def _case(kind, n, seed=0):
    """(oracle policy, fp32 flat theta, engine.load_policy kwargs, obs, act, adv) for one of the test policies."""
    g = torch.Generator().manual_seed(seed)
    if kind == "polA":
        ws = [torch.from_numpy(G[f"polA/w{i}"]) for i in range(3)]
        bs = [torch.from_numpy(G[f"polA/b{i}"]) for i in range(3)]
        ls = torch.from_numpy(G["polA/log_std"])
        tf, nl = {}, "tanh"
    elif kind == "polB":
        ws = [torch.from_numpy(G[f"polB/w{i}"]) for i in range(4)]
        bs = [torch.from_numpy(G[f"polB/b{i}"]) for i in range(4)]
        ls = torch.full((12,), -0.7)
        tf = dict(in_shift=G["polB/in_shift"], in_scale=G["polB/in_scale"], out_shift=G["polB/out_shift"],
                  out_scale=G["polB/out_scale"])
        nl = "relu"
    else:  # mjrl's default 64 x 64 relu policy on the MILO observation / action sizes
        sizes = [226, 64, 64, 28]
        ws = [torch.randn(o, i, generator=g) / i ** 0.5 for i, o in zip(sizes[:-1], sizes[1:])]
        bs = [torch.randn(o, generator=g) * 0.1 for o in sizes[1:]]
        ls = torch.full((28,), -0.5) + 0.1 * torch.randn(28, generator=g)
        tf, nl = {}, "relu"
    sizes = [ws[0].shape[1]] + [w.shape[0] for w in ws]
    pol = no.Policy(sizes, nl, **{k: torch.as_tensor(v) for k, v in tf.items()})
    theta = pol.flatten(ws, bs, ls).float()
    obs = torch.randn(n, sizes[0], generator=g)
    if kind == "polB":
        obs = obs * torch.as_tensor(G["polB/in_scale"]) + torch.as_tensor(G["polB/in_shift"])
    mu = pol.mean(theta.double(), obs).float()
    act = mu + torch.exp(ls) * torch.randn(n, sizes[-1], generator=g)
    adv = torch.randn(n, generator=g)
    kw = dict(weights=ws, biases=bs, nonlinearity=nl, log_std=ls, **tf)
    return pol, theta, kw, obs, act, adv


def _load(eng, kw, theta):
    eng.load_policy(kw["weights"], kw["biases"], kw["nonlinearity"], kw.get("in_shift"), kw.get("in_scale"),
                    kw.get("out_shift"), kw.get("out_scale"), kw["log_std"])
    eng.npg_init()
    eng.npg_params(theta.cuda())


def _rel(x, ref):
    ref = torch.as_tensor(ref, dtype=torch.float64)
    return float(torch.linalg.norm(torch.as_tensor(x, dtype=torch.float64).cpu() - ref) / torch.linalg.norm(ref))


@pytest.mark.parametrize("kind,n", [("polA", 4097), ("polB", 31), ("polB", 1), ("relu64", 4097), ("polA", 1)])
def test_gradient_and_fisher_vector_product_match_the_oracle(kind, n):
    eng = _engine()
    pol, theta, kw, obs, act, adv = _case(kind, n)
    _load(eng, kw, theta)
    P = pol.n_params
    o, a, d = obs.cuda(), act.cuda(), adv.cuda()
    gs = eng.npg_grad(o, a, d).cpu()
    assert gs[P] == n
    ref = no.vpg_grad(pol, theta.double(), obs, act, adv)
    assert _rel(gs[:P] / n, ref) < 1e-4
    assert abs(float(gs[P + 1]) - float(adv.double().sum())) < 1e-4 * max(1.0, float(adv.abs().sum()))
    v = torch.randn(P, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    eng.npg_prepare(o)
    fs = eng.npg_fvp(o, v=v.cuda()).cpu()
    assert fs[P] == n
    assert _rel(fs[:P] / n, no.hvp(pol, theta.double(), obs, v)) < 1e-4


def test_fisher_vector_product_at_rollout_size():
    """1.28 M rows (40 000 envs x 32 steps) of the MILO-sized policy: the sums over many CTAs stay within 1e-3."""
    eng = _engine()
    n = 40_000 * 32
    pol, theta, kw, obs, act, adv = _case("polA", n)
    _load(eng, kw, theta)
    P = pol.n_params
    o, a, d = obs.cuda(), act.cuda(), adv.cuda()
    gs = eng.npg_grad(o, a, d).cpu()
    ref = torch.zeros(P, dtype=torch.float64)
    v = torch.randn(P, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    href = torch.zeros(P, dtype=torch.float64)
    for s in range(0, n, 160_000):  # the oracle in row chunks (sums of means)
        sl = slice(s, s + 160_000)
        m = obs[sl].shape[0]
        ref += no.vpg_grad(pol, theta.double(), obs[sl], act[sl], adv[sl]) * m
        href += no.hvp(pol, theta.double(), obs[sl], v) * m
    eng.npg_prepare(o)
    fs = eng.npg_fvp(o, v=v.cuda()).cpu()
    assert _rel(gs[:P], ref) < 1e-3
    assert _rel(fs[:P], href) < 1e-3


class _HostPolicy:
    def __init__(self, kw, theta):
        class M:
            pass
        self.model = M()
        self.model.fc_layers = [torch.nn.Linear(w.shape[1], w.shape[0]) for w in kw["weights"]]
        for l, w, b in zip(self.model.fc_layers, kw["weights"], kw["biases"]):
            l.weight.data, l.bias.data = w.clone().float(), b.clone().float()
        self.model.nonlinearity = torch.relu if kw["nonlinearity"] == "relu" else torch.tanh
        obs, act = kw["weights"][0].shape[1], kw["weights"][-1].shape[0]
        self.model.in_shift = torch.as_tensor(kw.get("in_shift", np.zeros(obs, np.float32)))
        self.model.in_scale = torch.as_tensor(kw.get("in_scale", np.ones(obs, np.float32)))
        self.model.out_shift = torch.as_tensor(kw.get("out_shift", np.zeros(act, np.float32)))
        self.model.out_scale = torch.as_tensor(kw.get("out_scale", np.ones(act, np.float32)))
        self.log_std = torch.as_tensor(kw["log_std"]).clone().float()
        self.min_log_std = -3.0


@pytest.mark.parametrize("mode", ["plain", "valid", "subsample", "const_lr"])
def test_full_update_matches_the_oracle(mode):
    from amp_extensions_b200.npg import DeviceNPG
    eng = _engine()
    n = 6000
    pol, theta, kw, obs, act, adv = _case("polA", n, seed=2)
    adv = (adv - adv.mean()) / adv.std()
    host = _HostPolicy(kw, theta)
    opt = dict(cg_iters=10)
    if mode == "subsample":
        opt["hvp_sample_frac"] = 0.25
    if mode == "const_lr":
        opt["const_learn_rate"] = 0.05
    npg = DeviceNPG(eng, host, **opt)
    valid = None
    if mode == "valid":
        valid = (torch.rand(n, generator=torch.Generator().manual_seed(3)) < 0.7).to(torch.uint8)
    idx = None
    if mode == "subsample":   # the rows DeviceNPG will draw: same generator, same call
        gen = torch.Generator(device="cuda")
        gen.manual_seed(0)
        idx = torch.randint(0, n, (int(0.25 * n),), device="cuda", generator=gen, dtype=torch.int64).cpu()
    out = npg.update((obs.cuda(), act.cuda()), adv.cuda(), None if valid is None else valid.cuda())
    out = {k: float(v) for k, v in out.items()}
    new_ref, ref = no.npg_step(pol, theta.double(), obs, act, adv, valid=valid, fisher_idx=idx,
                               const_learn_rate=opt.get("const_learn_rate"), cg_iters=10, damping=1e-4)
    got = npg.params().cpu().double()
    assert _rel(got - theta.double(), new_ref - theta.double()) < 1e-3
    for k in ("alpha", "kl_dist", "surr_after", "surr_before"):
        assert abs(out[k] - ref[k]) <= 1e-3 * max(abs(ref[k]), 1e-6 if k != "surr_before" else 1e-3), (k, out[k], ref[k])
    assert out["cg_iters_run"] == ref["cg_iters_run"]


def test_updates_are_bit_identical_and_graph_capturable():
    from amp_extensions_b200.npg import DeviceNPG
    n = 20_000
    pol, theta, kw, obs, act, adv = _case("polA", n, seed=4)
    o, a, d = obs.cuda(), act.cuda(), adv.cuda()
    res = []
    for k in range(2):
        eng = _engine()
        npg = DeviceNPG(eng, _HostPolicy(kw, theta))
        out = npg.update((o, a), d)
        res.append((npg.params().clone(), {k2: v.clone() for k2, v in out.items()}))
    assert torch.equal(res[0][0], res[1][0])
    assert all(torch.equal(res[0][1][k], res[1][1][k]) for k in res[0][1])
    # the same update captured in a CUDA graph (after an eager warm-up update that sizes the workspaces)
    eng = _engine()
    npg = DeviceNPG(eng, _HostPolicy(kw, theta))
    npg.update((o, a), d)
    torch.cuda.synchronize()
    eng.npg_params(theta.cuda())
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            out = npg.update((o, a), d)
    torch.cuda.current_stream().wait_stream(s)
    eng.npg_params(theta.cuda())
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(npg.params(), res[0][0])
    assert all(torch.equal(out[k], res[0][1][k]) for k in out)


def test_update_writes_the_policy_in_place():
    """policy_act after update equals a fresh load_policy of the exported parameters; the engine generation is unchanged,
    so a collect(graph=True) graph captured before the update replays with the new policy."""
    from amp_extensions_b200 import AmpDataset, DynamicsEnsemble, HumanoidTermination, VecSimEnv
    from amp_extensions_b200.npg import DeviceNPG
    from amp_extensions_b200.rollout import DeviceRollout
    c = H.tiny_case("tiny_dense")
    S, A = c["S"], c["A"]
    s, a, s2 = c["ds"]
    ens = DynamicsEnsemble(S, A, AmpDataset(s, a, s2), None, num_models=c["N"], hidden_sizes=c["hidden"],
                           dense_connect=True, transform=True, base_seed=100)
    g = torch.Generator().manual_seed(0)
    kw = dict(weights=[torch.randn(16, S, generator=g) * 0.2, torch.randn(A, 16, generator=g) * 0.2],
              biases=[torch.zeros(16), torch.zeros(A)], nonlinearity="tanh", log_std=torch.full((A,), -1.0))
    host = _HostPolicy(kw, None)
    env = VecSimEnv(ens, 64, termination=HumanoidTermination(horizon=5, fall_contact_bodies=()), reset_states=s[:32], seed=0)
    env.reset(initial_states=s[:64])
    ro = DeviceRollout(env, host, seed=0)
    T = 6
    noise = torch.randn(T, 64, A, generator=g).cuda()
    pick = torch.randint(0, 32, (T, 64), generator=g, dtype=torch.int32).cuda()
    b = ro.collect(T, noise=noise, pick=pick, graph=True)
    npg = DeviceNPG(ro, host, normalized_step_size=0.05)
    gen0, n_graphs = ro.eng.generation, len(ro._graphs)
    adv = torch.randn(T * 64, generator=g).cuda()
    npg.update(b, adv)
    assert ro.eng.generation == gen0
    obs = torch.randn(300, S, generator=g).cuda()
    _, mean_new = ro.eng.policy_act(obs)
    eng_graph = ro._graphs[next(iter(ro._graphs))][0]
    theta = npg.export_params()
    fresh = _engine()
    fresh.load_policy([l.weight.data for l in host.model.fc_layers], [l.bias.data for l in host.model.fc_layers], "tanh",
                      log_std=host.log_std)
    _, mean_ref = fresh.policy_act(obs)
    assert torch.equal(mean_new, mean_ref)
    act_new, _ = ro.eng.policy_act(obs, torch.ones(300, A, device="cuda"))
    act_ref, _ = fresh.policy_act(obs, torch.ones(300, A, device="cuda"))
    assert torch.allclose(act_new, act_ref, rtol=2e-7, atol=0)   # std within an ulp
    # the cached rollout graph is replayed (not re-captured) and runs the new policy
    env.reset(initial_states=s[:64])
    b2 = ro.collect(T, noise=noise, pick=pick, graph=True)
    assert len(ro._graphs) == n_graphs and ro._graphs[next(iter(ro._graphs))][0] is eng_graph
    _, m0 = fresh.policy_act(b2.observations[0].contiguous())
    assert torch.equal(b2.means[0], m0)
    assert theta.numel() == npg.n_params


def test_oversized_policy_is_rejected():
    from amp_extensions_b200 import _lib
    eng = _engine()
    ws = [torch.zeros(96, 226), torch.zeros(96, 96), torch.zeros(28, 96)]
    eng.load_policy(ws, [torch.zeros(96), torch.zeros(96), torch.zeros(28)], "tanh", log_std=torch.zeros(28))
    with pytest.raises(_lib.SimstepError, match="does not fit"):
        eng.npg_init()


def test_debug_guards_after_an_update(monkeypatch):
    monkeypatch.setenv("SIMSTEP_DEBUG_GUARDS", "1")
    from amp_extensions_b200.npg import DeviceNPG
    eng = _engine()
    pol, theta, kw, obs, act, adv = _case("polB", 3001)
    npg = DeviceNPG(eng, _HostPolicy(kw, theta), hvp_sample_frac=0.5)
    npg.update((obs.cuda(), act.cuda()), adv.cuda(), (torch.arange(3001) % 3 != 0).to(torch.uint8).cuda())
    n_buf, bad = eng.check_guards()
    assert n_buf >= 10 and bad == 0


def test_milo_iteration_with_npg_steps():
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples"))
    import milo_iteration
    out, _ = milo_iteration.main(num_envs=256, horizon=24, epochs=1, n_offline=2048, verbose=False, npg_steps=3)
    assert len(out["npg"]) == 3
    for it in out["npg"]:
        assert it["surr_after"] > it["surr_before"], it
        assert it["kl_dist"] <= 0.01, it


def _nccl_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    from amp_extensions_b200 import parallel
    from amp_extensions_b200.npg import DeviceNPG
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    device = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=device)
    pol, theta, kw, obs, act, adv = _case("polA", 9001, seed=7)
    a, b = parallel.shard_range(obs.shape[0])
    npg = DeviceNPG(_engine(), _HostPolicy(kw, theta))
    out = npg.update((obs[a:b].to(device), act[a:b].to(device)), adv[a:b].to(device))
    torch.save(dict(theta=npg.params().cpu(), **{k: float(v) for k, v in out.items()}), os.path.join(out_dir, f"rank{rank}.pt"))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_gpu_row_sharded_update_equals_single_gpu():
    import socket
    import tempfile
    import torch.multiprocessing as mp
    from amp_extensions_b200.npg import DeviceNPG
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    with tempfile.TemporaryDirectory() as d:
        mp.spawn(_nccl_worker, args=(2, port, d), nprocs=2, join=True)
        parts = [torch.load(os.path.join(d, f"rank{r}.pt"), weights_only=False) for r in range(2)]
    pol, theta, kw, obs, act, adv = _case("polA", 9001, seed=7)
    npg = DeviceNPG(_engine(), _HostPolicy(kw, theta))
    out = {k: float(v) for k, v in npg.update((obs.cuda(), act.cuda()), adv.cuda()).items()}
    ref = npg.params().cpu().double()
    for p in parts:
        assert torch.equal(p["theta"], parts[0]["theta"])
        assert _rel(p["theta"].double() - theta.double(), ref - theta.double()) < 1e-5
        for k in ("alpha", "kl_dist", "surr_after"):
            assert abs(p[k] - out[k]) <= 1e-5 * abs(out[k]), k


def test_engine_changes_other_than_the_policy_keep_the_device_parameters():
    """A generation bump that does not replace the policy (termination, cost, ensemble changes) must not reset the NPG
    state to the host object's stale values: two updates with a set_termination in between equal two updates without,
    bit for bit, and the rollout engine's generation is not bumped by the update itself."""
    from amp_extensions_b200 import HumanoidTermination
    from amp_extensions_b200.npg import DeviceNPG
    pol, theta, kw, obs, act, adv = _case("polA", 5000, seed=5)
    o, a, d = obs.cuda(), act.cuda(), adv.cuda()
    res = []
    for bump in (False, True):
        eng = _engine()
        npg = DeviceNPG(eng, _HostPolicy(kw, theta))
        npg.update((o, a), d)
        after_one = npg.params().clone()
        if bump:
            gen = eng.generation
            eng.set_termination(HumanoidTermination(horizon=7, fall_contact_bodies=()))
            assert eng.generation == gen + 1
        npg.update((o, a), d)
        if bump:
            assert eng.generation == gen + 1
        res.append((after_one, npg.params().clone()))
    assert not torch.equal(res[1][0], theta.cuda()) and not torch.equal(res[1][1], res[1][0])
    assert torch.equal(res[0][1], res[1][1])
    # a load_policy of the host object does re-attach: the next update starts from the host values again
    eng = _engine()
    host = _HostPolicy(kw, theta)
    npg = DeviceNPG(eng, host)
    npg.update((o, a), d)
    _load(eng, kw, theta)
    npg.update((o, a), d)
    assert torch.equal(npg.params(), res[0][0])


def test_update_converts_host_rows_and_engine_calls_refuse_them():
    from amp_extensions_b200.npg import DeviceNPG
    pol, theta, kw, obs, act, adv = _case("polA", 3000, seed=6)
    eng = _engine()
    npg = DeviceNPG(eng, _HostPolicy(kw, theta))
    out_host = {k: v.clone() for k, v in npg.update((obs.double(), act), adv.double()).items()}
    p_host = npg.params().clone()
    eng.npg_params(theta.cuda())
    out_dev = npg.update((obs.cuda(), act.cuda()), adv.cuda())
    assert torch.equal(npg.params(), p_host) and all(torch.equal(out_dev[k], out_host[k]) for k in out_dev)
    with pytest.raises(TypeError):
        eng.npg_grad(obs, act.cuda(), adv.cuda())
    with pytest.raises(TypeError):
        eng.npg_fvp(obs.cuda().double())
    with pytest.raises(ValueError):
        npg.update((obs.cuda(), act[:10].cuda()), adv.cuda())


def test_fvp_sums_write_a_zero_advantage_slot():
    eng = _engine()
    pol, theta, kw, obs, act, adv = _case("polB", 257)
    _load(eng, kw, theta)
    o = obs.cuda()
    eng.npg_prepare(o)
    out = torch.full((pol.n_params + 2,), float("nan"), device="cuda", dtype=torch.float64)
    eng.npg_fvp(o, v=torch.ones(pol.n_params, device="cuda", dtype=torch.float64), out=out)
    assert float(out[-2]) == 257 and float(out[-1]) == 0.0 and bool(torch.isfinite(out).all())


def test_export_goes_through_set_param_values_when_the_policy_has_it():
    from amp_extensions_b200.npg import DeviceNPG, flat_params

    class MjrlLike(_HostPolicy):
        def __init__(self, kw, theta):
            super().__init__(kw, theta)
            self.calls = []

        def set_param_values(self, new_params, set_new=True, set_old=True):
            self.calls.append((np.array(new_params), set_new, set_old))
            self.log_std_val = np.asarray(new_params)[-len(self.log_std):].astype(np.float64)

    pol, theta, kw, obs, act, adv = _case("polA", 2000, seed=8)
    host = MjrlLike(kw, theta)
    npg = DeviceNPG(_engine(), host)
    npg.update((obs.cuda(), act.cuda()), adv.cuda())
    t = npg.export_params()
    assert len(host.calls) == 1 and host.calls[0][1:] == (True, True)
    assert np.array_equal(host.calls[0][0], t.numpy()) and not torch.equal(t, flat_params(host))
