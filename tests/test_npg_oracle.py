"""The NPG oracle (oracle/npg_oracle.py) against the reference's pinned policy outputs and against itself: the
double-autograd HVP equals the closed-form Fisher and finite differences, CG matches a dense solve, the step's KL follows
the quadratic model, the min_log_std clamp, and the flat parameter order of an mjrl-shaped policy object."""
import os

import numpy as np
import torch

from oracle import npg_oracle as no

G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "rollout_golden.npz"))


def golden_policy(tag, n_layers, log_std=None):
    ws = [G[f"{tag}/w{i}"] for i in range(n_layers)]
    bs = [G[f"{tag}/b{i}"] for i in range(n_layers)]
    sizes = [ws[0].shape[1]] + [w.shape[0] for w in ws]
    kw = {}
    if tag == "polB":
        kw = dict(in_shift=G["polB/in_shift"], in_scale=G["polB/in_scale"], out_shift=G["polB/out_shift"],
                  out_scale=G["polB/out_scale"])
    pol = no.Policy(sizes, "tanh" if tag == "polA" else "relu", **kw)
    ls = G["polA/log_std"] if log_std is None else log_std
    return pol, pol.flatten(ws, bs, ls)


def small_case(seed=0, n=64, sizes=(5, 6, 3), nl="tanh"):
    g = torch.Generator().manual_seed(seed)
    pol = no.Policy(sizes, nl, in_shift=torch.randn(sizes[0], generator=g, dtype=torch.float64) * 0.1,
                    in_scale=1 + torch.rand(sizes[0], generator=g, dtype=torch.float64),
                    out_shift=torch.randn(sizes[-1], generator=g, dtype=torch.float64) * 0.1,
                    out_scale=0.5 + torch.rand(sizes[-1], generator=g, dtype=torch.float64))
    theta = torch.randn(pol.n_params, generator=g, dtype=torch.float64) * 0.5
    theta[-sizes[-1]:] = -0.5 + 0.1 * torch.randn(sizes[-1], generator=g, dtype=torch.float64)
    obs = torch.randn(n, sizes[0], generator=g, dtype=torch.float64)
    act = pol.mean(theta, obs) + torch.exp(theta[-sizes[-1]:]) * torch.randn(n, sizes[-1], generator=g, dtype=torch.float64)
    adv = torch.randn(n, generator=g, dtype=torch.float64)
    return pol, theta, obs, act, adv


def test_oracle_mean_equals_reference_policy_outputs():
    pol, theta = golden_policy("polA", 3)
    ref = G["polA/mean"]
    assert np.abs(pol.mean(theta, G["polA/obs"]).numpy() - ref).max() <= 2e-6 * np.abs(ref).max()
    pol, theta = golden_policy("polB", 4, log_std=np.zeros(12, np.float32))
    ref = G["polB/mean"]
    assert np.abs(pol.mean(theta, G["polB/obs"]).numpy() - ref).max() <= 2e-6 * np.abs(ref).max()


def test_hvp_equals_closed_form_fisher_and_finite_differences():
    for nl in ("tanh", "relu"):
        pol, theta, obs, _, _ = small_case(1, nl=nl)
        v = torch.randn(pol.n_params, generator=torch.Generator().manual_seed(2), dtype=torch.float64)
        hv = no.hvp(pol, theta, obs, v)
        F = no.fisher_closed_form(pol, theta, obs)
        assert torch.allclose(hv, F @ v, rtol=1e-10, atol=1e-12)
        # finite differences of grad mean_kl(., theta) around theta
        def grad_kl(t):
            t = t.clone().requires_grad_(True)
            return torch.autograd.grad(pol.mean_kl(t, theta, obs), t)[0]
        h = 1e-6
        fd = (grad_kl(theta + h * v) - grad_kl(theta - h * v)) / (2 * h)
        assert torch.linalg.norm(fd - hv) <= 1e-6 * torch.linalg.norm(hv)


def test_cg_matches_dense_solve():
    pol, theta, obs, act, adv = small_case(3)
    damping = 1e-4
    g = no.vpg_grad(pol, theta, obs, act, adv)
    F = no.fisher_closed_form(pol, theta, obs) + damping * torch.eye(pol.n_params, dtype=torch.float64)
    x, it = no.cg_solve(lambda v: F @ v, g, cg_iters=3 * pol.n_params, residual_tol=1e-30)
    ref = torch.linalg.solve(F, g)
    assert torch.linalg.norm(x - ref) <= 1e-6 * torch.linalg.norm(ref)


def test_vanilla_gradient_closed_form():
    """d LL / d mu_j = z_j / s_j, d LL / d log_std_j = z_j^2 - 1."""
    pol, theta, obs, act, adv = small_case(4)
    g = no.vpg_grad(pol, theta, obs, act, adv)
    A = pol.sizes[-1]
    s = torch.exp(theta[-A:])
    z = (act - pol.mean(theta, obs)) / s
    assert torch.allclose(g[-A:], (adv[:, None] * (z ** 2 - 1)).mean(0), rtol=1e-10, atol=1e-12)
    J = torch.func.jacrev(lambda t: pol.mean(t, obs))(theta)
    ref = torch.einsum("na,nap->p", adv[:, None] * z / s, J) / obs.shape[0]
    assert torch.allclose(g[:-A], ref[:-A], rtol=1e-10, atol=1e-12)


def test_step_kl_follows_the_quadratic_model():
    pol, theta, obs, act, adv = small_case(5, n=256)
    delta = 1e-4
    new, out = no.npg_step(pol, theta.float().double(), obs, act, adv, normalized_step_size=delta,
                           cg_iters=4 * pol.n_params, damping=1e-4)
    assert abs(out["kl_dist"] - delta / 2) <= 0.05 * delta / 2
    assert out["surr_after"] > out["surr_before"]


def test_min_log_std_clamp():
    pol, theta, obs, act, adv = small_case(6)
    pol.min_log_std = float(theta[-3:].min()) + 1e-3
    new, out = no.npg_step(pol, theta, obs, act, adv, const_learn_rate=0.0)
    assert float(new[-3:].min()) >= pol.min_log_std - 1e-7
    assert torch.equal(new[:-3], theta[:-3].float().double())


def test_flat_order_round_trips_through_an_mjrl_shaped_policy():
    from amp_extensions_b200.npg import flat_params, set_flat_params

    class Model:
        pass

    class MLP:
        def __init__(self, sizes):
            self.model = Model()
            self.model.fc_layers = [torch.nn.Linear(i, o) for i, o in zip(sizes[:-1], sizes[1:])]
            self.log_std = torch.nn.Parameter(torch.full((sizes[-1],), -0.5))
            self.trainable_params = [p for l in self.model.fc_layers for p in l.parameters()] + [self.log_std]
            self.min_log_std = -3.0

    pi = MLP([5, 6, 3])
    theta = flat_params(pi)
    ref = torch.cat([p.detach().reshape(-1) for p in pi.trainable_params])
    assert torch.equal(theta, ref)
    pol = no.Policy([5, 6, 3])
    ws, bs, ls = pol.unflatten(theta.double())
    for w, l in zip(ws, pi.model.fc_layers):
        assert torch.equal(w.float(), l.weight.detach())
    new = torch.arange(theta.numel(), dtype=torch.float32) * -0.01
    set_flat_params(pi, new, pi.min_log_std)
    got = flat_params(pi)
    assert torch.equal(got[:-3], new[:-3]) and torch.equal(got[-3:], torch.clamp(new[-3:], min=-3.0))
    # a policy without trainable_params: fc_layers weight / bias pairs, then log_std
    class Bare:
        pass
    b = Bare()
    b.model = Model()
    b.model.fc_layers = pi.model.fc_layers
    b.log_std = pi.log_std.detach().clone()
    assert torch.equal(flat_params(b), got)
