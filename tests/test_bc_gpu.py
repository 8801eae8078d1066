"""Behaviour cloning on the GPU (csrc/bc.cuh, csrc/bc_api.inc, amp_extensions_b200/bc.py) against the float64 oracle
(oracle/bc_oracle.py) at every policy shape tests/test_policy_matrix_gpu.py loads (L = 1 - 4, widths 1 - 128, obs_dim
1 - 512, act_dim 1 - 128, tanh and relu, with and without transforms; relu rows clear the mask margin there), both
losses, batch sizes 1, 63, 64, 65, 256 and 1024 and index tables with duplicates: the full-data loss, one step's
gradient per tensor, the Adam update, fits of 200 steps and of a whole 1 000 000-row epoch, the in-place commit into
the policy (rollout graphs, the NPG state), reproducibility, graph replay, isolation, refusals and the guard zones.

Worst values measured on one B200 (1 000 W power limit) / asserted bounds:
  full-data loss, both losses      relative                                    1.6e-8 / 3e-8
  forward against policy_act       RMS of the mean, of the largest |mean|      1.1e-7 / 4e-6
  one step's gradient              weight, of the tensor's largest entry       1.2e-6 / 2.5e-6
                                   bias                                        9.1e-6 / 2e-5
                                   log_std (MLE)                               4.0e-6 / 8e-6
  200-step fit (tanh)              parameters, of the largest |parameter|      1.6e-5 / 3.5e-5
  200-step fit (relu)              parameters                                  1.7e-3 / 3.5e-3
  200-step fit                     loss_after relative                         1.6e-6 / 4e-6
  1 000 000 rows, one epoch        loss_after relative                         1.8e-6 / 5e-6
  NPG step after the fit           relative L2 of the step                     1.9e-6 / 1e-3 (test_policy_matrix_gpu's)
The bias bound is set by act_dim = 1 (blocks1537): the output bias gradient is one sum of residuals of both signs, so
the fp32 forward's rounding shows relative to a small total.  In a relu fit a unit whose pre-activation crosses zero
flips its mask a step earlier or later in fp32 than in fp64, which moves the parameters apart (the loss still agrees to
1.6e-6); the tanh fits bound the parameters tightly.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import bc_oracle as bo
from oracle import npg_oracle as no
from tests import test_policy_matrix_gpu as M

BOUND = {"loss": 3e-8, "grad": {"weight": 2.5e-6, "bias": 2e-5, "log_std": 8e-6}, "fit_params": 3.5e-5,
         "fit_params_relu": 3.5e-3, "fit_loss": 4e-6, "full_loss": 5e-6}
IDS = M.IDS + [c["id"] for c in M.REFUSED]   # BC has no per-CTA accumulator limit: NPG's refused shapes load too
BATCHES = [1, 63, 64, 65, 256, 1024]
LOSSES = ["MSE", "MLE"]


def _setup(cid, loss, bs, epochs=1, **kw):
    from amp_extensions_b200.bc import DeviceBC
    cd = M.case_data(cid)
    eng = M.engine()
    M.load(eng, cd)
    host = M.host_policy(cd, cd["theta"])
    bc = DeviceBC(eng, host, epochs=epochs, batch_size=bs, loss_type=loss, **kw)
    return cd, eng, host, bc


def _rows(cd, n=None):
    obs, act = cd["obs"], cd["act"]
    if n is not None:
        obs, act = obs[:n], act[:n]
    return obs.contiguous(), act.contiguous()


def _table(n, steps, bs, seed):
    g = torch.Generator().manual_seed(seed)
    idx = torch.randint(0, n, (steps, bs), generator=g)
    idx[0, -1] = idx[0, 0]   # a row drawn twice counts twice
    return idx


@pytest.mark.gpu
@pytest.mark.parametrize("cid", IDS)
def test_full_data_loss_matches_the_oracle(cid):
    cd, eng, host, bc = _setup(cid, "MSE", 64)
    obs, act = _rows(cd)
    pol, theta = cd["pol"], cd["theta"].double()
    worst = 0.0
    for loss in LOSSES:
        bc.loss_type = loss
        bc._attach()
        got = float(bc.loss(obs.cuda(), act.cuda()))
        with torch.no_grad():
            ref = float(bo.loss(loss, pol, bo.params_of(pol, theta), obs, act))
        e = abs(got - ref) / abs(ref)
        worst = max(worst, e)
        assert e <= BOUND["loss"], (cid, loss, got, ref)
    # MSE against policy_act's own mean: the two forwards agree (RMS within test_policy_matrix_gpu's 4e-6 of the
    # largest |mean|)
    bc.loss_type = "MSE"
    bc._attach()
    _, mean = eng.policy_act(obs.cuda())
    rms = float(bc.loss(obs.cuda(), mean)) ** 0.5
    print(f"loss {cid}: worst {worst:.2e}; forward vs policy_act rms {rms / float(mean.abs().max()):.2e}")
    assert rms <= M.REL["mean"] * float(mean.abs().max())


@pytest.mark.gpu
@pytest.mark.parametrize("loss", LOSSES)
@pytest.mark.parametrize("cid", IDS)
def test_one_step_gradient_matches_the_oracle(cid, loss):
    cd, eng, host, bc = _setup(cid, loss, 64)
    obs, act = _rows(cd)
    n = obs.shape[0]
    o, a = obs.cuda(), act.cuda()
    pol, theta = cd["pol"], cd["theta"]
    worst = {}
    for bs in BATCHES:
        eng.bc_init(bs, loss, theta)
        idx = _table(n, 1, bs, seed=bs)
        eng.bc_fit(o, a, idx.reshape(-1).cuda(), 1)
        st = eng.bc_read()
        assert st["step"] == 1
        ref = bo.minibatch_grads(loss, pol, theta.double(), obs, act, idx[0])
        M.check_parts(pol, st["grad"].cpu(), ref, BOUND["grad"], (cid, loss, bs), worst)
        if loss == "MSE":
            assert torch.equal(st["params"][-pol.sizes[-1]:].cpu(), theta[-pol.sizes[-1]:])
    print(f"grad {cid} {loss}: " + ", ".join(f"{k} {v:.2e}" for k, v in worst.items()))


@pytest.mark.gpu
@pytest.mark.parametrize("loss", LOSSES)
def test_adam_update_matches_a_float32_restatement(loss):
    """One step from an imported Adam state (step 5, non-zero moments, weight decay 0.1), from the gradient the device
    computed; MSE leaves log_std and both of its moments bit-identical."""
    cd = M.case_data("polA")
    lr, wd, b1, b2, eps = 3e-3, 0.1, 0.9, 0.999, 1e-8
    eng = M.engine()
    M.load(eng, cd)
    P = cd["pol"].n_params
    g = torch.Generator().manual_seed(4)
    m0, v0 = 1e-2 * torch.randn(P, generator=g), 1e-4 * torch.rand(P, generator=g)
    eng.bc_init(64, loss, cd["theta"], lr=lr, weight_decay=wd, exp_avg=m0, exp_avg_sq=v0, step=5)
    s0 = eng.bc_read()
    obs, act = _rows(cd, 640)
    eng.bc_fit(obs.cuda(), act.cuda(), torch.arange(640, device="cuda"), 1)
    s1 = eng.bc_read()
    f32 = np.float32
    cnt = P if loss == "MLE" else P - cd["pol"].sizes[-1]
    w, m, v, gr = (s0["params"].cpu().numpy(), s0["exp_avg"].cpu().numpy(), s0["exp_avg_sq"].cpu().numpy(),
                   s1["grad"].cpu().numpy())
    fma = lambda a, b, c: f32(np.float64(a) * np.float64(b) + np.float64(c))
    gw = fma(f32(wd), w, gr)
    m1 = fma(f32(b1), m, (f32(1) - f32(b1)) * gw)
    v1 = fma(f32(b2), v, (f32(1) - f32(b2)) * gw * gw)
    bc1, bc2 = f32(1.0 - float(f32(b1)) ** 6), f32(1.0 - float(f32(b2)) ** 6)
    w1 = fma(-(f32(lr) / bc1), m1 / (np.sqrt(v1) / np.sqrt(bc2) + f32(eps)), w)
    for name, got, want, old in (("exp_avg", s1["exp_avg"], m1, m), ("exp_avg_sq", s1["exp_avg_sq"], v1, v),
                                 ("params", s1["params"], w1, w)):
        got = got.cpu().numpy()
        ulps = np.abs(got[:cnt] - want[:cnt]) / np.spacing(np.abs(want[:cnt]))
        print(f"{loss} {name}: worst {ulps.max():.2f} ulp")
        assert ulps.max() <= 1.0, name
        np.testing.assert_array_equal(got[cnt:], old[cnt:])   # MSE: log_std and its moments untouched
    assert s1["step"] == 6


def _oracle_fit(cd, loss, theta, obs, act, idx, epochs, bs, device="cpu"):
    pol = cd["pol"]
    if device != "cpu":
        pol = no.Policy(pol.sizes, pol.nonlinearity, *(t.to(device) for t in (pol.in_shift, pol.in_scale,
                                                                                pol.out_shift, pol.out_scale)),
                        min_log_std=pol.min_log_std)
    params = [p.detach().to(device).requires_grad_(True) for p in bo.params_of(pol, theta.double().cpu())]
    before, after = bo.fit(pol, params, bo.make_adam(params, loss), obs.to(device).double(), act.to(device).double(),
                           idx.to(device), epochs, bs, loss)
    return before, after, bo.flat(params).cpu()


@pytest.mark.gpu
@pytest.mark.parametrize("cid, bs", [("polA", 64), ("relu_tf", 32)])
@pytest.mark.parametrize("loss", LOSSES)
def test_a_200_step_fit_tracks_the_oracle(cid, bs, loss):
    cd, eng, host, bc = _setup(cid, loss, bs)
    n = 200 * bs
    obs, act = _rows(cd, n)
    idx = _table(n, 200, bs, seed=7)
    before, after = bc.fit_tensors(obs.cuda(), act.cuda(), idx=idx, return_losses=True)
    rb, ra, p_ref = _oracle_fit(cd, loss, cd["theta"], obs, act, idx, 1, bs)
    p_dev = bc.params().double().cpu()
    perr = float((p_dev - p_ref).abs().max() / p_ref.abs().max())
    eb, ea = abs(float(before) - rb) / abs(rb), abs(float(after) - ra) / abs(ra)
    print(f"200-step {cid} {loss}: loss_before rel {eb:.2e}, loss_after {float(after):.6e} (oracle {ra:.6e}, rel "
          f"{ea:.2e}), parameters {perr:.2e}")
    pb = BOUND["fit_params_relu" if cd["pol"].nonlinearity == "relu" else "fit_params"]
    assert eb <= BOUND["loss"] and ea <= BOUND["fit_loss"] and perr <= pb and ra < rb


@pytest.mark.gpu
@pytest.mark.parametrize("loss", LOSSES)
def test_full_epoch_at_1000000_rows(loss):
    """The MILO policy (226 -> 32 -> 32 -> 28 tanh), batch 64, one epoch of 15 625 steps on 1 000 000 rows whose
    actions are a teacher policy's mean plus noise; the oracle runs in float64 on the same GPU."""
    bs, n = 64, 1_000_000
    cd, eng, host, bc = _setup("polA", loss, bs)
    g = torch.Generator().manual_seed(11)
    obs = torch.randn(n, 226, generator=g)
    teacher = cd["pol"].n_params
    t_theta = torch.randn(teacher, generator=g, dtype=torch.float64) * 0.2
    with torch.no_grad():
        act = (cd["pol"].mean(t_theta, obs) + 0.1 * torch.randn(n, 28, generator=g, dtype=torch.float64)).float()
    idx = torch.randint(0, n, (n // bs, bs), generator=g)
    before, after = bc.fit_tensors(obs.cuda(), act.cuda(), idx=idx, return_losses=True)
    rb, ra, _ = _oracle_fit(cd, loss, cd["theta"], obs, act, idx, 1, bs, device="cuda")
    eb, ea = abs(float(before) - rb) / abs(rb), abs(float(after) - ra) / abs(ra)
    print(f"1M rows {loss}: loss_before rel {eb:.2e}, loss_after {float(after):.6e} (oracle {ra:.6e}, rel {ea:.2e})")
    assert eb <= BOUND["loss"] and ea <= BOUND["full_loss"] and float(after) < float(before)


@pytest.mark.gpu
def test_mse_leaves_log_std_alone_and_export_writes_no_state_for_it():
    cd, eng, host, bc = _setup("polA", "MSE", 64)
    obs, act = _rows(cd, 6400)
    A = 28
    bc.fit_tensors(obs.cuda(), act.cuda())
    st = eng.bc_read()
    assert torch.equal(st["params"][-A:].cpu(), cd["theta"][-A:])
    assert float(st["exp_avg"][-A:].abs().max()) == 0 and float(st["exp_avg_sq"][-A:].abs().max()) == 0
    bc.export()
    assert host.log_std not in bc.optimizer.state and len(bc.optimizer.state) == len(bc.optimizer.param_groups[0]["params"]) - 1
    assert int(float(bc.optimizer.state[host.model.fc_layers[0].weight]["step"])) == 100


@pytest.mark.gpu
def test_mle_moves_log_std_and_commit_clamps_it():
    cd = M.case_data("polA")
    from amp_extensions_b200.bc import DeviceBC
    eng = M.engine()
    M.load(eng, cd)
    theta = cd["theta"].clone()
    theta[-28:] = -0.55
    host = M.host_policy(cd, theta)
    host.min_log_std = -0.6
    M.load(eng, dict(cd, kw=dict(cd["kw"], log_std=theta[-28:])))
    bc = DeviceBC(eng, host, epochs=3, batch_size=64, loss_type="MLE", lr=1e-2)
    obs, act = _rows(cd, 6400)
    mu = eng.policy_act(obs.cuda())[1]
    mu = mu + 1e-3 * torch.randn(mu.shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(0))
    bc.fit_tensors(obs.cuda(), mu)
    ls = bc.params()[-28:]
    assert bool((ls == np.float32(-0.6)).all()), ls
    # the handle's std tail: a fresh load of the exported parameters samples the same actions
    noise = torch.randn(obs.shape[0], 28, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
    _check_pack_equals_fresh_load(eng, cd, bc, obs.cuda(), noise)


def _check_pack_equals_fresh_load(eng, cd, bc, obs, noise):
    theta = bc.export()
    ws, bs_, ls = cd["pol"].unflatten(theta.double())
    fresh = M.engine()
    kw = cd["kw"]
    fresh.load_policy([w.float() for w in ws], [b.float() for b in bs_], kw["nonlinearity"], kw.get("in_shift"),
                      kw.get("in_scale"), kw.get("out_shift"), kw.get("out_scale"), ls.float())
    a1, m1 = eng.policy_act(obs, noise)
    a2, m2 = fresh.policy_act(obs, noise)
    assert torch.equal(a1, a2) and torch.equal(m1, m2)


@pytest.mark.gpu
@pytest.mark.parametrize("cid", ["polA", "relu_tf", "linear"])
def test_commit_is_in_place_for_graphs_and_matches_a_fresh_load(cid):
    cd, eng, host, bc = _setup(cid, "MLE", 64)
    obs, act = _rows(cd, 4096)
    o = obs.cuda()
    noise = torch.randn(4096, cd["pol"].sizes[-1], device="cuda", generator=torch.Generator(device="cuda").manual_seed(2))
    act_out, mean_out = eng.policy_act(o, noise)
    before = act_out.clone()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()   # what a DeviceRollout graph captures of the policy
    with torch.cuda.graph(graph):
        eng.policy_act(o, noise, action=act_out, mean=mean_out)
    gen = eng.generation
    bc.fit_tensors(o, act.cuda())
    assert eng.generation == gen
    graph.replay()
    a_eager, m_eager = eng.policy_act(o, noise)
    assert torch.equal(act_out, a_eager) and torch.equal(mean_out, m_eager) and not torch.equal(before, act_out)
    _check_pack_equals_fresh_load(eng, cd, bc, o, noise)


@pytest.mark.gpu
@pytest.mark.parametrize("loss", LOSSES)
def test_npg_built_before_the_fit_steps_from_the_cloned_parameters(loss):
    from amp_extensions_b200.npg import DeviceNPG
    cd, eng, host, bc = _setup("polA", loss, 64)
    npg = DeviceNPG(eng, M.host_policy(cd, cd["theta"]))
    n = 6000
    obs, act = _rows(cd, n)
    adv = cd["adv"][:n]
    adv = (adv - adv.mean()) / adv.std()
    idx = _table(n, n // 64, 64, seed=3)
    bc.fit_tensors(obs.cuda(), act.cuda(), idx=idx)
    _, _, p_ref = _oracle_fit(cd, loss, cd["theta"], obs, act, idx, 1, 64)
    theta_bc = bc.params().double().cpu()
    assert float((theta_bc - p_ref).abs().max() / p_ref.abs().max()) <= BOUND["fit_params"]
    assert torch.equal(npg.params().cpu(), bc.params().cpu())
    npg.update((obs.cuda(), act.cuda()), adv.cuda())
    want, _ = no.npg_step(cd["pol"], theta_bc, obs, act, adv)
    got = npg.params().double().cpu()
    err = M.rel_l2(got - theta_bc, want - theta_bc)
    print(f"NPG after BC {loss}: step relative L2 {err:.2e}")
    assert err <= M.UPDATE_REL


@pytest.mark.gpu
def test_zero_steps_leave_the_parameters_bit_identical():
    cd, eng, host, bc = _setup("polA", "MLE", 64)
    p0 = bc.params().clone()
    for n in (63, 1, 0):
        obs, act = _rows(cd, n)
        before, after = bc.fit_tensors(obs.cuda(), act.cuda(), return_losses=True)
        assert torch.equal(bc.params(), p0) and eng.bc_read()["step"] == 0
        if n:
            assert np.isfinite(float(before)) and float(before) == float(after)
        else:
            assert np.isnan(float(before)) and np.isnan(float(after))


@pytest.mark.gpu
def test_two_fits_are_bit_identical_and_graph_replay_matches_eager():
    cd, eng, host, bc = _setup("polA", "MLE", 64)
    obs, act = _rows(cd, 4096)
    o, a = obs.cuda(), act.cuda()
    nb = 4096 // 64
    idx = _table(4096, nb, 64, seed=5).reshape(-1).cuda()
    s0 = {k: (v.clone() if torch.is_tensor(v) else v) for k, v in eng.bc_read().items()}

    def restore():
        eng.bc_state(params=s0["params"], exp_avg=s0["exp_avg"], exp_avg_sq=s0["exp_avg_sq"], step=s0["step"])

    def state():
        return {k: (v.clone() if torch.is_tensor(v) else v) for k, v in eng.bc_read().items()}
    eng.bc_fit(o, a, idx, nb)
    first = state()
    restore()
    eng.bc_fit(o, a, idx, nb)
    second = state()
    assert first["step"] == second["step"] == nb
    for k in ("params", "exp_avg", "exp_avg_sq", "grad"):
        assert torch.equal(first[k], second[k]), k
    restore()
    torch.cuda.synchronize()
    g_epoch = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g_epoch):
        eng.bc_fit(o, a, idx, nb)
    g_epoch.replay()
    s = state()
    assert s["step"] == nb and all(torch.equal(s[k], first[k]) for k in ("params", "exp_avg", "exp_avg_sq"))
    restore()
    torch.cuda.synchronize()
    g_first, g_next = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
    with torch.cuda.graph(g_first):
        eng.bc_fit(o, a, idx, 7, restart=True)
    with torch.cuda.graph(g_next):
        eng.bc_fit(o, a, idx, 7, restart=False)
    g_first.replay()
    for _ in range(nb // 7 + 2):   # the last replays run past the epoch's end: no-ops
        g_next.replay()
    s = state()
    assert s["step"] == nb and all(torch.equal(s[k], first[k]) for k in ("params", "exp_avg", "exp_avg_sq"))


@pytest.mark.gpu
def test_ensemble_cost_and_baseline_loads_leave_the_state_alone_and_load_policy_drops_it():
    from amp_extensions_b200 import _lib
    from amp_extensions_b200.baseline import DeviceMLPBaseline, MLPBaseline
    from tests import helpers as H
    cd, eng, host, bc = _setup("polA", "MLE", 64)
    obs, act = _rows(cd, 2048)
    o, a = obs.cuda(), act.cuda()
    idx = _table(2048, 32, 64, seed=9).reshape(-1).cuda()
    eng.bc_fit(o, a, idx, 3)
    s1 = {k: (v.clone() if torch.is_tensor(v) else v) for k, v in eng.bc_read().items()}
    case = H.tiny_case("tiny_dense")
    eng.load_ensemble(case["ws"], case["bs"], case["tf"])
    g = torch.Generator().manual_seed(0)
    eng.load_rff(torch.randn(64, case["S"], generator=g), torch.rand(64, generator=g), input_type="s")

    class Spec:
        observation_dim = 17
    DeviceMLPBaseline(eng, MLPBaseline(Spec(), hidden_sizes=(8,)))
    s2 = eng.bc_read()
    assert s2["step"] == s1["step"] and all(torch.equal(s1[k], s2[k]) for k in ("params", "exp_avg", "exp_avg_sq"))
    eng.bc_fit(o, a, idx, 100, restart=False)   # the epoch continues where it stopped
    assert eng.bc_read()["step"] == 32
    M.load(eng, cd)
    with pytest.raises(_lib.SimstepError):
        eng.bc_read()
    before, after = bc.fit_tensors(o, a, return_losses=True)   # re-attaches from the host policy
    assert eng.bc_read()["step"] == 32 and float(after) < float(before)


@pytest.mark.gpu
def test_a_smaller_bc_on_another_handle_leaves_the_first_running():
    cd, eng, host, bc = _setup("obs512", "MLE", 1024)
    obs, act = _rows(cd, 4096)
    o, a = obs.cuda(), act.cuda()
    idx = _table(4096, 4, 1024, seed=1).reshape(-1).cuda()
    s0 = {k: (v.clone() if torch.is_tensor(v) else v) for k, v in eng.bc_read().items()}
    loss0 = float(bc.loss(o, a))
    eng.bc_fit(o, a, idx, 4)
    fitted = eng.bc_read()["params"].clone()
    cd2, eng2, _, bc2 = _setup("obs1", "MSE", 1)
    o2, a2 = _rows(cd2, 64)
    bc2.fit_tensors(o2.cuda(), a2.cuda())
    eng.bc_state(params=s0["params"], exp_avg=s0["exp_avg"], exp_avg_sq=s0["exp_avg_sq"], step=s0["step"])
    assert float(bc.loss(o, a)) == loss0
    eng.bc_fit(o, a, idx, 4)
    assert torch.equal(eng.bc_read()["params"], fitted)


@pytest.mark.gpu
def test_refusals_leave_the_handle_usable():
    import ctypes as C
    from amp_extensions_b200 import _lib
    from amp_extensions_b200 import engine as E
    cd = M.case_data("polA")
    eng = M.engine()
    with pytest.raises(_lib.SimstepError, match="load_policy"):
        eng.bc_init(64, "MSE", cd["theta"])
    M.load(eng, cd)
    theta = cd["theta"].cuda()
    for bs in (0, 1025):
        with pytest.raises(_lib.SimstepError, match="batch_size"):
            eng.bc_init(bs, "MSE", theta)
    with pytest.raises(_lib.SimstepError, match="loss type"):
        eng._check(eng.lib.simstep_bc_init(eng._h, 64, 7, 1e-3, 0.9, 0.999, 1e-8, 0.0, -3.0, E._ptr(theta), None, None,
                                           0, None))
    eng.bc_init(64, "MLE", theta)
    obs, act = _rows(cd, 256)
    o, a = obs.cuda(), act.cuda()
    out = torch.empty(3, device="cuda", dtype=torch.float64)
    with pytest.raises(_lib.SimstepError, match="n < 0"):
        eng._check(eng.lib.simstep_bc_loss(eng._h, E._ptr(o), E._ptr(a), -1, E._ptr(out), E._stream(eng.device)))
    with pytest.raises(_lib.SimstepError, match="n < 0"):
        eng._check(eng.lib.simstep_bc_fit(eng._h, E._ptr(o), E._ptr(a), -1, E._ptr(out), 64, 1, 1,
                                          E._stream(eng.device)))
    eng.bc_fit(o, a, torch.arange(256, device="cuda"), 4)
    assert eng.bc_read()["step"] == 4 and np.isfinite(float(eng.bc_loss(o, a)[1]))


GUARD_SCRIPT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "write_bc_guards.py")


@pytest.mark.gpu
def test_guard_zones_around_bc_buffers(tmp_path):
    """Guarded BC buffers: theta, grad, m, v, x, the log_std terms, dz_l per layer, h_l per hidden layer, the Adam
    state, the cursor, the descriptor, the loss partials and pack_of."""
    out = str(tmp_path / "guards.npz")
    env = dict(os.environ, SIMSTEP_DEBUG_GUARDS="1")
    res = subprocess.run([sys.executable, GUARD_SCRIPT, out], env=env, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-3000:]
    z = np.load(out)
    for cid in IDS:
        n0, n1, bad = z[cid]
        L = len(M.CASE[cid]["sizes"]) - 1
        assert n1 - n0 == 10 + 2 * L and bad == 0, (cid, n0, n1, bad)


@pytest.mark.gpu
def test_milo_iteration_with_a_bc_warm_start(monkeypatch):
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples"))
    import milo_iteration
    from amp_extensions_b200.bc import DeviceBC
    from amp_extensions_b200.rollout import DeviceRollout
    seen = {}
    collect, fit = DeviceRollout.collect, DeviceBC.fit_tensors

    def collect_first(self, *a, **k):
        batch = collect(self, *a, **k)
        seen.setdefault("first", (batch.observations[0].clone(), batch.means[0].clone()))
        return batch

    def fit_and_keep(self, *a, **k):
        res = fit(self, *a, **k)
        seen["theta"] = self.params().clone()
        return res
    monkeypatch.setattr(DeviceRollout, "collect", collect_first)
    monkeypatch.setattr(DeviceBC, "fit_tensors", fit_and_keep)
    out, _ = milo_iteration.main(num_envs=256, horizon=24, epochs=1, n_offline=2048, verbose=False, bc_epochs=2)
    b, a = out["bc_loss_before"], out["bc_loss_after"]
    print(f"milo_iteration bc_epochs=2: bc_loss_before {b:.4e}, bc_loss_after {a:.4e}")
    assert np.isfinite(b) and np.isfinite(a) and a < b
    obs, mean = seen["first"]
    pol = no.Policy((226, 32, 32, 28), "tanh")
    ref = pol.mean(seen["theta"].double().cpu(), obs.double().cpu())
    assert M.rel_to_max(mean.cpu(), ref) <= M.REL["mean"]
