"""The MLP value baseline on the GPU (csrc/baseline.cuh, amp_extensions_b200/baseline.py) against the float64 oracle
(oracle/baseline_oracle.py): features, predict, one step's gradients, the Adam update with weight decay, whole fits,
reproducibility, graph replay, independence from the handle's other components, and the workspace guard zones.

Shapes: hidden (), (32,), (128, 128), (256, 256), (64, 64, 64); obs_dim 1, 17, 226, 512; rows 1, 63, 64, 65, 129,
6 144; batch sizes 1, 64, 256, and cases that leave zero optimiser steps (n < 2 * batch_size).

Worst values measured on one B200 (1 000 W power limit) / asserted bounds:
  predict                      relative to the largest |value|          2.5e-7 / 1e-5
  one step's gradients         per tensor, of its largest entry          1.6e-7 / 1e-5
  200-step fit (S = 226)       error_before relative                    9.7e-11 / 1e-5
                               error_after relative                      7.0e-9 / 1e-7
                               parameters, of the largest |parameter|    1.1e-6 / 3e-6
  40 000 x 32 rows, one epoch  error_before relative                    3.7e-11 / 1e-5
                               error_after relative                      8.0e-3 / 3e-2
The 19 999-step fit is chaotic: fp32 and fp64 trajectories separate (the parameters end up O(1) apart, as two fp32
torch runs with different summation orders do), while the fitted error agrees to about 1 %.
"""
import numpy as np
import pytest
import torch

from oracle import baseline_oracle as bo

FIT_ERR_BOUND = 1e-7
FIT_PARAM_BOUND = 3e-6
FULL_ERR_BOUND = 3e-2

CASES = [  # hidden, obs_dim, rows, batch_size
    ((), 1, 63, 1),
    ((32,), 17, 129, 64),
    ((128, 128), 226, 6144, 64),
    ((256, 256), 512, 65, 1),
    ((64, 64, 64), 226, 6144, 256),
    ((128, 128), 17, 64, 64),      # zero steps
    ((32,), 512, 1, 1),            # zero steps, one row
    ((), 226, 6144, 256),
    ((64, 64, 64), 17, 65, 1),
    ((256, 256), 1, 129, 256),     # zero steps
]


def _engine():
    from amp_extensions_b200.engine import Engine
    return Engine(state_dim=8, action_dim=0, num_models=1, hidden_sizes=[], transform=False)


def _host(S, hidden, bs, lr=1e-3, wd=0.0, epochs=1, seed=0):
    from amp_extensions_b200.baseline import MLPBaseline

    class Spec:
        observation_dim = S

    torch.manual_seed(seed)
    return MLPBaseline(Spec(), learn_rate=lr, reg_coef=wd, batch_size=bs, epochs=epochs, hidden_sizes=hidden)


def _paths(n, S, seed, max_len=1500, lengths=()):
    """Paths of random lengths (t up to max_len - 1; the first ones of the given lengths) with observations partly
    beyond +-10; returns a smooth function of the features plus noise."""
    rng = np.random.default_rng(seed)
    paths, left, lengths = [], n, list(lengths)
    while left > 0:
        l = int(min(left, lengths.pop(0) if lengths else rng.integers(1, max_len + 1)))
        obs = rng.standard_normal((l, S)) * 6.0
        obs = obs.astype(np.float32).astype(np.float64)
        ret = (np.tanh(obs[:, : min(S, 5)]).sum(1) + 0.3 * rng.standard_normal(l) + np.arange(l) / 500.0)
        paths.append({"observations": obs, "rewards": np.zeros(l), "returns": ret})
        left -= l
    return paths


def _device_rows(paths):
    obs = torch.from_numpy(np.concatenate([p["observations"] for p in paths]).astype(np.float32)).cuda()
    t = torch.from_numpy(np.concatenate([np.arange(len(p["rewards"])) for p in paths]).astype(np.int32)).cuda()
    y = torch.from_numpy(np.concatenate([p["returns"] for p in paths]).astype(np.float32)).cuda()
    return obs.contiguous(), t.contiguous(), y.contiguous()


def _model64(vf, params=None):
    return bo.make_model(vf.sizes, (vf.eng.baseline_read()["params"] if params is None else params).double().cpu())


def _tensors(sizes, v):
    out, off = [], 0
    for i, o in zip(sizes[:-1], sizes[1:]):
        for k in (o * i, o):
            out.append(v[off:off + k])
            off += k
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("S", [1, 17, 226, 512])
def test_device_features_equal_the_oracles_float32_features(S):
    """Read column j of the device's features through a one-layer net with the one-hot weight e_j and no bias: the
    fp32 sum of x_j and exact zeros is x_j."""
    from amp_extensions_b200.baseline import DeviceMLPBaseline
    eng = _engine()
    vf = DeviceMLPBaseline(eng, _host(S, (), 64))
    paths = _paths(1300, S, seed=S, lengths=[1200]) + _paths(40, S, seed=S + 1, max_len=40)
    obs, t, _ = _device_rows(paths)
    ref = bo.features_f32(paths)
    got = np.empty_like(ref)
    for j in range(S + 4):
        w = torch.zeros(S + 5)
        w[j] = 1.0
        eng.baseline_state(params=w)
        got[:, j] = eng.baseline_predict(obs, t).cpu().numpy()
    np.testing.assert_array_equal(got[:, :S], ref[:, :S])
    assert np.all(np.abs(got[:, S:] - ref[:, S:]) <= np.spacing(np.abs(ref[:, S:]))), "time columns beyond 1 ulp"
    assert np.abs(ref[:, :S]).max() == 1.0 and float(ref[:, S].max()) > 1.0  # clipping and t >= 1000 were exercised


@pytest.mark.gpu
@pytest.mark.parametrize("hidden, S, n, bs", CASES)
def test_predict_matches_the_float64_oracle(hidden, S, n, bs):
    from amp_extensions_b200.baseline import DeviceMLPBaseline
    vf = DeviceMLPBaseline(_engine(), _host(S, hidden, bs, seed=n))
    paths = _paths(n, S, seed=n + S)
    obs, t, _ = _device_rows(paths)
    got = vf.eng.baseline_predict(obs, t).double().cpu()
    ref = bo.predict(_model64(vf), bo.features_f32(paths))
    err = float((got - ref).abs().max() / ref.abs().max())
    print(f"predict {hidden} S={S} n={n}: {err:.2e}")
    assert err <= 1e-5
    if n > 1:
        np.testing.assert_array_equal(vf.predict(paths[0]), got[:len(paths[0]["rewards"])].float().numpy())


@pytest.mark.gpu
def test_predict_batch_equals_predict_on_the_batchs_paths():
    from amp_extensions_b200.baseline import DeviceMLPBaseline
    from amp_extensions_b200.rollout import RolloutBatch
    eng = _engine()
    T, E, S, A = 40, 64, 17, 3
    vf = DeviceMLPBaseline(eng, _host(S, (32,), 64))
    b = RolloutBatch(eng, T, E, S, A, False)
    g = torch.Generator(device="cuda").manual_seed(0)
    for x in (b.observations, b.next_observations, b.actions, b.means, b.disc):
        x.normal_(generator=g)
    b.observations.mul_(8.0)
    b.done.copy_((torch.rand(T, E, device="cuda", generator=g) < 0.08).to(torch.uint8))
    b.done[:, 0] = 0
    b.rewards = torch.zeros(T, E, device="cuda")
    b.log_std = torch.zeros(A, device="cuda")
    pred = vf.predict_batch(b).cpu().numpy()
    assert pred.shape == (T, E)
    for (e, t0, t1, _), path in zip(b.segments(), b.paths()):
        np.testing.assert_array_equal(vf.predict(path), pred[t0:t1, e])


@pytest.mark.gpu
@pytest.mark.parametrize("hidden, S, n, bs", CASES)
def test_one_step_gradients_match_the_float64_oracle(hidden, S, n, bs):
    from amp_extensions_b200.baseline import DeviceMLPBaseline
    eng = _engine()
    vf = DeviceMLPBaseline(eng, _host(S, hidden, bs, seed=n))
    paths = _paths(n, S, seed=2 * n + S)
    obs, t, y = _device_rows(paths)
    p0 = eng.baseline_read()
    perm = torch.randperm(n, device="cuda", generator=torch.Generator(device="cuda").manual_seed(n))
    eng.baseline_fit(obs, t, y, perm, n_steps=1)
    st = eng.baseline_read()
    if bo.num_batches(n, bs) == 0:   # fit_data takes no step: nothing changes, not even the step count
        assert st["step"] == 0 and torch.equal(st["params"], p0["params"]) and torch.equal(st["exp_avg"], p0["exp_avg"])
        return
    idx = perm[:bs].cpu().numpy()
    x = bo.features_f32(paths)[idx]
    ref = bo.minibatch_grads(_model64(vf, p0["params"]), x, y.cpu().numpy()[idx])
    worst = 0.0
    for g_dev, g_ref in zip(_tensors(vf.sizes, st["grad"].double().cpu()), _tensors(vf.sizes, ref)):
        scale = float(g_ref.abs().max())
        if scale > 0:
            worst = max(worst, float((g_dev - g_ref).abs().max()) / scale)
    print(f"grad {hidden} S={S} n={n} bs={bs}: {worst:.2e}")
    assert st["step"] == 1 and worst <= 1e-5


@pytest.mark.gpu
def test_adam_update_with_weight_decay_matches_a_float32_restatement():
    """One step from an imported Adam state (step 5, non-zero moments) with reg_coef = 0.1: the update kernel against
    its float32 restatement, from the gradient the device computed."""
    from amp_extensions_b200.baseline import DeviceMLPBaseline
    S, bs, lr, wd, b1, b2, eps = 17, 64, 3e-3, 0.1, 0.9, 0.999, 1e-8
    host = _host(S, (32,), bs, lr=lr, wd=wd)
    g = torch.Generator().manual_seed(4)
    for p in host.model.parameters():
        host.optimizer.state[p] = {"step": torch.tensor(5.0), "exp_avg": 1e-2 * torch.randn(p.shape, generator=g),
                                   "exp_avg_sq": 1e-4 * torch.rand(p.shape, generator=g)}
    eng = _engine()
    vf = DeviceMLPBaseline(eng, host)
    s0 = eng.baseline_read()
    assert s0["step"] == 5
    obs, t, y = _device_rows(_paths(200, S, seed=9))
    eng.baseline_fit(obs, t, y, torch.arange(200, device="cuda"), n_steps=1)
    s1 = eng.baseline_read()
    f32 = np.float32
    w, m, v, gr = (s0["params"].cpu().numpy(), s0["exp_avg"].cpu().numpy(), s0["exp_avg_sq"].cpu().numpy(),
                   s1["grad"].cpu().numpy())
    fma = lambda a, b, c: f32(np.float64(a) * np.float64(b) + np.float64(c))
    gw = fma(f32(wd), w, gr)
    m1 = fma(f32(b1), m, (f32(1) - f32(b1)) * gw)
    v1 = fma(f32(b2), v, (f32(1) - f32(b2)) * gw * gw)
    bc1, bc2 = f32(1.0 - float(f32(b1)) ** 6), f32(1.0 - float(f32(b2)) ** 6)   # fp32 betas, fp64 powers
    w1 = fma(-(f32(lr) / bc1), m1 / (np.sqrt(v1) / np.sqrt(bc2) + f32(eps)), w)   # w -= lr' * x contracts to one fma
    for name, got, want in (("exp_avg", s1["exp_avg"], m1), ("exp_avg_sq", s1["exp_avg_sq"], v1),
                            ("params", s1["params"], w1)):
        got = got.cpu().numpy()
        ulps = np.abs(got - want) / np.spacing(np.abs(want))
        i = int(np.argmax(ulps))
        print(f"{name}: worst {ulps[i]:.2f} ulp at {i}: {got[i]!r} vs {want[i]!r} (w {w[i]!r}, g {gr[i]!r})")
        assert ulps[i] <= 1.0, name
    assert s1["step"] == 6 and not np.array_equal(s1["params"].cpu().numpy(), w)


def _fit_against_oracle(S, hidden, n, bs, seed, oracle_device="cpu"):
    from amp_extensions_b200.baseline import DeviceMLPBaseline
    eng = _engine()
    vf = DeviceMLPBaseline(eng, _host(S, hidden, bs, seed=seed))
    paths = _paths(n, S, seed=seed, max_len=32)
    obs, t, y = _device_rows(paths)
    perm = torch.randperm(n, device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed))
    model = _model64(vf).to(oracle_device)
    before, after = vf._fit(obs, t, y, None, True, perm)
    x = torch.from_numpy(bo.features_f32(paths)).to(oracle_device)
    yy = y.to(oracle_device)
    ref_before = bo.error(model, x, yy)
    bo.fit(model, bo.make_adam(model), x, yy, [perm.to(oracle_device)], bs)
    ref_after = bo.error(model, x, yy)
    p_dev, p_ref = eng.baseline_read()["params"].double().cpu(), bo.flat(model).cpu()
    return (float(before), float(after), ref_before, ref_after,
            float((p_dev - p_ref).abs().max() / p_ref.abs().max()))


@pytest.mark.gpu
def test_a_200_step_fit_tracks_the_oracle():
    bs = 64
    before, after, rb, ra, perr = _fit_against_oracle(226, (128, 128), bs * 201, bs, seed=7)
    e_before, e_after = abs(before - rb) / rb, abs(after - ra) / ra
    print(f"200-step fit: error_before {before:.6e} (oracle {rb:.6e}, rel {e_before:.2e}), error_after {after:.6e} "
          f"(oracle {ra:.6e}, rel {e_after:.2e}), parameters {perr:.2e}")
    assert e_before <= 1e-5 and e_after <= FIT_ERR_BOUND and perr <= FIT_PARAM_BOUND and after < before


@pytest.mark.gpu
def test_full_size_epoch_at_40000_by_32_rows():
    """The reference's default network (230 -> 128 -> 128 -> 1, batch 64, one epoch: 19 999 Adam steps) on
    40 000 x 32 rows; the oracle runs in float64 on the same GPU."""
    before, after, rb, ra, perr = _fit_against_oracle(226, (128, 128), 40_000 * 32, 64, seed=11, oracle_device="cuda")
    e_before, e_after = abs(before - rb) / rb, abs(after - ra) / ra
    print(f"40000x32 fit: error_before {before:.6e} (oracle {rb:.6e}, rel {e_before:.2e}), error_after {after:.6e} "
          f"(oracle {ra:.6e}, rel {e_after:.2e}), parameters {perr:.2e}")
    assert e_before <= 1e-5 and e_after <= FULL_ERR_BOUND and after < before


def _state(eng):
    return {k: (v.clone() if torch.is_tensor(v) else v) for k, v in eng.baseline_read().items()}


def _restore(eng, s):
    eng.baseline_state(params=s["params"], exp_avg=s["exp_avg"], exp_avg_sq=s["exp_avg_sq"], step=s["step"])


@pytest.mark.gpu
def test_two_fits_from_the_same_state_are_bit_identical_and_graph_replay_matches_eager():
    from amp_extensions_b200.baseline import DeviceMLPBaseline
    eng = _engine()
    S, bs, n = 226, 64, 4096
    DeviceMLPBaseline(eng, _host(S, (128, 128), bs, wd=1e-4))
    obs, t, y = _device_rows(_paths(n, S, seed=3, max_len=64))
    perm = torch.randperm(n, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    nb = bo.num_batches(n, bs)
    s0 = _state(eng)
    eng.baseline_fit(obs, t, y, perm, nb)
    first = _state(eng)
    _restore(eng, s0)
    eng.baseline_fit(obs, t, y, perm, nb)
    second = _state(eng)
    assert first["step"] == second["step"] == nb
    for k in ("params", "exp_avg", "exp_avg_sq", "grad"):
        assert torch.equal(first[k], second[k]), k
    # a whole epoch captured into one graph (the capture fails if the epoch synchronises with the host)
    _restore(eng, s0)
    torch.cuda.synchronize()
    g_epoch = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g_epoch):
        eng.baseline_fit(obs, t, y, perm, nb)
    g_epoch.replay()
    s = _state(eng)
    assert s["step"] == nb and all(torch.equal(s[k], first[k]) for k in ("params", "exp_avg", "exp_avg_sq"))
    # chunks of 7 steps: a restarting chunk, then continuing chunks replayed past the end of the epoch (no-ops)
    _restore(eng, s0)
    torch.cuda.synchronize()
    g_first, g_next = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
    with torch.cuda.graph(g_first):
        eng.baseline_fit(obs, t, y, perm, 7, restart=True)
    with torch.cuda.graph(g_next):
        eng.baseline_fit(obs, t, y, perm, 7, restart=False)
    g_first.replay()
    for _ in range(nb // 7 + 2):
        g_next.replay()
    s = _state(eng)
    assert s["step"] == nb and all(torch.equal(s[k], first[k]) for k in ("params", "exp_avg", "exp_avg_sq"))


@pytest.mark.gpu
def test_loading_a_policy_or_an_ensemble_leaves_the_baseline_alone():
    from amp_extensions_b200.baseline import DeviceMLPBaseline
    from amp_extensions_b200.engine import Engine
    eng = Engine(state_dim=8, action_dim=2, num_models=2, hidden_sizes=[16], transform=False)
    g = torch.Generator().manual_seed(0)
    ens = ([[torch.randn(16, 10, generator=g), torch.randn(8, 16, generator=g)] for _ in range(2)],
           [[torch.randn(16, generator=g), torch.randn(8, generator=g)] for _ in range(2)])
    eng.load_ensemble(*ens)
    S = 226
    vf = DeviceMLPBaseline(eng, _host(S, (128, 128), 64))
    obs, t, y = _device_rows(_paths(1000, S, seed=5))
    perm = torch.randperm(1000, device="cuda", generator=torch.Generator(device="cuda").manual_seed(5))
    eng.baseline_fit(obs, t, y, perm, 3)
    s1 = _state(eng)
    pred = eng.baseline_predict(obs, t).clone()
    eng.load_policy([torch.randn(16, 8, generator=g), torch.randn(2, 16, generator=g)],
                    [torch.zeros(16), torch.zeros(2)], "tanh", log_std=torch.zeros(2))
    eng.npg_init()
    eng.load_ensemble(*ens)
    assert torch.equal(eng.baseline_predict(obs, t), pred)
    s2 = _state(eng)
    assert s2["step"] == s1["step"] and all(torch.equal(s1[k], s2[k]) for k in ("params", "exp_avg", "exp_avg_sq"))
    eng.baseline_fit(obs, t, y, perm, 100, restart=False)   # the epoch continues where it stopped
    assert eng.baseline_read()["step"] == bo.num_batches(1000, 64)


@pytest.mark.gpu
def test_a_smaller_baseline_on_another_handle_leaves_the_first_running():
    from amp_extensions_b200.baseline import DeviceMLPBaseline
    a, b = _engine(), _engine()
    DeviceMLPBaseline(a, _host(512, (256, 256), 256))
    obs, t, y = _device_rows(_paths(2048, 512, seed=1))
    perm = torch.arange(2048, device="cuda")
    first = a.baseline_predict(obs, t).clone()
    s0 = _state(a)
    a.baseline_fit(obs, t, y, perm, 7)
    fitted = _state(a)
    DeviceMLPBaseline(b, _host(1, (), 1))
    ob, tb, yb = _device_rows(_paths(64, 1, seed=2))
    b.baseline_predict(ob, tb)
    b.baseline_fit(ob, tb, yb, torch.arange(64, device="cuda"), 62)
    _restore(a, s0)
    assert torch.equal(a.baseline_predict(obs, t), first)
    a.baseline_fit(obs, t, y, perm, 7)
    assert torch.equal(a.baseline_read()["params"], fitted["params"])


@pytest.mark.gpu
def test_refusals_leave_the_handle_usable():
    from amp_extensions_b200 import _lib
    eng = _engine()
    ok = dict(batch_size=64, params=torch.zeros(7 * 4 + 4 + 5))
    for sizes, bs in (((7, 4, 1), 0), ((7, 4, 1), 1025), ((4, 1), 64), ((517, 1), 64), ((7, 257, 1), 64),
                      ((7, 4, 2), 64), ((7, 4, 4, 4, 4, 1), 64)):
        with pytest.raises(_lib.SimstepError):
            eng.baseline_init(sizes, bs, torch.zeros(10))
    eng.baseline_init((7, 4, 1), **ok)
    assert eng.baseline_predict(torch.zeros(3, 3, device="cuda"), torch.zeros(3, dtype=torch.int32, device="cuda")
                                ).abs().max() == 0
    # the reference default (230 -> 128 -> 128 -> 1, batch 64) and the largest supported shape are accepted
    eng.baseline_init((230, 128, 128, 1), 64, torch.zeros(230 * 128 + 128 + 128 * 128 + 128 + 129))
    eng.baseline_init((516, 256, 256, 256, 1), 1024, torch.zeros(516 * 256 + 2 * 256 * 257 + 256 + 257))


@pytest.mark.gpu
def test_guard_zones_stay_intact(monkeypatch):
    from amp_extensions_b200.baseline import DeviceMLPBaseline
    monkeypatch.setenv("SIMSTEP_DEBUG_GUARDS", "1")
    for hidden, S, n, bs in ((((64, 64, 64), 226, 6144, 256)), ((), 512, 129, 1), ((256, 256), 17, 2000, 1024)):
        eng = _engine()
        vf = DeviceMLPBaseline(eng, _host(S, hidden, bs, epochs=2))
        obs, t, y = _device_rows(_paths(n, S, seed=n))
        vf._fit(obs, t, y, None, True, None)
        eng.baseline_predict(obs, t)
        torch.cuda.synchronize()
        buffers, bad = eng.check_guards()
        assert buffers > 0 and bad == 0, (hidden, S, buffers, bad)


@pytest.mark.gpu
def test_milo_iteration_with_the_value_baseline():
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples"))
    import milo_iteration
    out, _ = milo_iteration.main(num_envs=256, horizon=24, epochs=1, n_offline=2048, verbose=False, vf_epochs=2)
    b, a = out["vf_error_before"], out["vf_error_after"]
    print(f"milo_iteration vf_epochs=2: vf_error_before {b:.4e}, vf_error_after {a:.4e}")
    assert np.isfinite(b) and np.isfinite(a) and a < b
    assert abs(out["adv_mean"]) < 1e-5 and abs(out["adv_std"] - 1.0) < 1e-4
