"""CPU oracle of the NPG policy step — TEST INFRASTRUCTURE, NOT PRODUCT CODE.

A float64 torch-autograd restatement of mjrl's NPG.train_from_paths (mjrl/mjrl/algos/npg_cg.py) on the Gaussian MLP
policy (mjrl/mjrl/policies/gaussian_mlp.py, mjrl/mjrl/utils/fc_network.py) with cg_solve (mjrl/mjrl/utils/cg_solve.py):

  LL        = -1/2 sum_j z_j^2 - sum_j log_std_j - A/2 log(2 pi),  z = (a - mu) / exp(log_std)
  g         = grad mean(exp(LL_new - LL_old) adv) at new = old
  F v       = Hessian of mean_kl(new, old) at new = old, times v, + damping v      (double autograd)
  x         = cg_solve(F, g, cg_iters): x = 0, r = p = g, stop when r.r < 1e-10
  alpha     = sqrt(|delta / (g.x + 1e-10)|)  or a fixed learning rate
  theta_new = theta + alpha x, log_std clamped at min_log_std (set_param_values)
  surr_after = mean(exp(LL_new - LL_old) adv),  kl_dist = mean_kl(new, old)

The parameter vector is in get_param_values order: per linear layer weight [out][in] then bias, then log_std.
"""
import math

import numpy as np
import torch


class Policy:
    """Shapes and fixed parts (transformations, nonlinearity) of a policy; parameters come as a flat vector."""

    def __init__(self, sizes, nonlinearity="tanh", in_shift=None, in_scale=None, out_shift=None, out_scale=None,
                 min_log_std=-3.0):
        self.sizes = list(sizes)
        self.nonlinearity = nonlinearity
        d = torch.float64
        obs, act = self.sizes[0], self.sizes[-1]
        self.in_shift = torch.zeros(obs, dtype=d) if in_shift is None else torch.as_tensor(in_shift, dtype=d)
        self.in_scale = torch.ones(obs, dtype=d) if in_scale is None else torch.as_tensor(in_scale, dtype=d)
        self.out_shift = torch.zeros(act, dtype=d) if out_shift is None else torch.as_tensor(out_shift, dtype=d)
        self.out_scale = torch.ones(act, dtype=d) if out_scale is None else torch.as_tensor(out_scale, dtype=d)
        self.min_log_std = float(min_log_std)

    @property
    def n_params(self):
        return sum(o * i + o for i, o in zip(self.sizes[:-1], self.sizes[1:])) + self.sizes[-1]

    def unflatten(self, theta):
        ws, bs, off = [], [], 0
        for i, o in zip(self.sizes[:-1], self.sizes[1:]):
            ws.append(theta[off:off + o * i].reshape(o, i)); off += o * i
            bs.append(theta[off:off + o]); off += o
        return ws, bs, theta[off:]

    def flatten(self, ws, bs, log_std):
        parts = []
        for w, b in zip(ws, bs):
            parts += [torch.as_tensor(w, dtype=torch.float64).reshape(-1), torch.as_tensor(b, dtype=torch.float64).reshape(-1)]
        parts.append(torch.as_tensor(np.asarray(log_std), dtype=torch.float64).reshape(-1))
        return torch.cat(parts)

    def mean(self, theta, obs):
        """FCNetwork.forward (fc_network.py:42-55) in float64."""
        ws, bs, _ = self.unflatten(theta)
        act = torch.relu if self.nonlinearity == "relu" else torch.tanh
        h = (torch.as_tensor(obs, dtype=torch.float64) - self.in_shift) / (self.in_scale + 1e-8)
        for w, b in zip(ws[:-1], bs[:-1]):
            h = act(h @ w.T + b)
        return (h @ ws[-1].T + bs[-1]) * self.out_scale + self.out_shift

    def log_likelihood(self, theta, obs, act):
        mu = self.mean(theta, obs)
        log_std = self.unflatten(theta)[2]
        z = (torch.as_tensor(act, dtype=torch.float64) - mu) / torch.exp(log_std)
        return -0.5 * (z ** 2).sum(dim=1) - log_std.sum() - 0.5 * mu.shape[1] * math.log(2 * math.pi)

    def mean_kl(self, theta_new, theta_old, obs):
        """MLP.mean_kl: mean_n sum_j ((mu_o - mu_n)^2 + s_o^2 - s_n^2) / (2 s_n^2 + 1e-8) + log s_n - log s_o."""
        mn, mo = self.mean(theta_new, obs), self.mean(theta_old, obs)
        ln, lo = self.unflatten(theta_new)[2], self.unflatten(theta_old)[2]
        sn, so = torch.exp(ln), torch.exp(lo)
        kl = ((mo - mn) ** 2 + so ** 2 - sn ** 2) / (2 * sn ** 2 + 1e-8) + ln - lo
        return kl.sum(dim=1).mean()


def _rows(x, valid):
    x = torch.as_tensor(x, dtype=torch.float64)
    return x if valid is None else x[torch.as_tensor(valid).bool()]


def surrogate(pol, theta_new, theta_old, obs, act, adv):
    """NPG.CPI_surrogate: mean(exp(LL_new - LL_old) adv)."""
    lr = torch.exp(pol.log_likelihood(theta_new, obs, act) - pol.log_likelihood(theta_old, obs, act))
    return (lr * torch.as_tensor(adv, dtype=torch.float64)).mean()


def vpg_grad(pol, theta, obs, act, adv):
    """NPG.flat_vpg: gradient of the surrogate at new = old."""
    t = theta.detach().clone().requires_grad_(True)
    s = surrogate(pol, t, theta.detach(), obs, act, adv)
    return torch.autograd.grad(s, t)[0]


def hvp(pol, theta, obs, v, damping=0.0):
    """NPG.HVP: Hessian of mean_kl(new, old) at new = old times v (double autograd), plus damping v."""
    t = theta.detach().clone().requires_grad_(True)
    kl = pol.mean_kl(t, theta.detach(), obs)
    g = torch.autograd.grad(kl, t, create_graph=True)[0]
    return torch.autograd.grad((g * torch.as_tensor(v, dtype=torch.float64)).sum(), t)[0] + damping * v


def fisher_closed_form(pol, theta, obs):
    """The same Hessian from the closed form: mean block (1/n) sum_n J_n^T diag(2 / (2 s^2 + eps)) J_n with J_n the
    Jacobian of the mean, log_std block diag(4 s^2 (2 s^2 - eps) / (2 s^2 + eps)^2), eps = 1e-8."""
    obs = torch.as_tensor(obs, dtype=torch.float64)
    J = torch.func.jacrev(lambda t: pol.mean(t, obs))(theta.detach())        # [n, A, P]
    s2 = torch.exp(2 * pol.unflatten(theta)[2])
    D = 2.0 / (2 * s2 + 1e-8)
    F = torch.einsum("naj,a,nak->jk", J, D, J) / obs.shape[0]
    ls0 = pol.n_params - pol.sizes[-1]
    F[ls0:, ls0:] += torch.diag(4 * s2 * (2 * s2 - 1e-8) / (2 * s2 + 1e-8) ** 2)
    return F


def cg_solve(f_Ax, b, cg_iters=10, residual_tol=1e-10):
    """mjrl/mjrl/utils/cg_solve.py: x = 0, r = p = b.  Returns (x, iterations run)."""
    x = torch.zeros_like(b)
    r = b.clone()
    p = r.clone()
    rdotr = r.dot(r)
    if rdotr == 0:
        return x, 0
    it = 0
    for _ in range(cg_iters):
        z = f_Ax(p)
        v = rdotr / p.dot(z)
        x = x + v * p
        r = r - v * z
        newrdotr = r.dot(r)
        p = r + (newrdotr / rdotr) * p
        rdotr = newrdotr
        it += 1
        if rdotr < residual_tol:
            break
    return x, it


def npg_step(pol, theta, obs, act, adv, valid=None, fisher_idx=None, normalized_step_size=0.01, const_learn_rate=None,
             cg_iters=10, damping=1e-4):
    """One NPG.train_from_paths policy step.  fisher_idx: rows of the HVP subsample (indices into all rows; rows masked
    out by `valid` do not count).  Returns (theta_new, dict(alpha, kl_dist, surr_before, surr_after, cg_iters_run, g, x))."""
    theta = torch.as_tensor(theta, dtype=torch.float64)
    obs_a, act_a, adv_a = (torch.as_tensor(x, dtype=torch.float64) for x in (obs, act, adv))
    if fisher_idx is not None:
        fi = torch.as_tensor(fisher_idx).long()
        keep = torch.ones(len(fi), dtype=torch.bool) if valid is None else torch.as_tensor(valid).bool()[fi]
        obs_f = obs_a[fi][keep]
    else:
        obs_f = _rows(obs_a, valid)
    obs_v, act_v, adv_v = _rows(obs_a, valid), _rows(act_a, valid), _rows(adv_a, valid)
    g = vpg_grad(pol, theta, obs_v, act_v, adv_v)
    x, it = cg_solve(lambda v: hvp(pol, theta, obs_f, v, damping), g, cg_iters)
    gx = float(g.dot(x))
    alpha = float(const_learn_rate) if const_learn_rate is not None else math.sqrt(abs(normalized_step_size / (gx + 1e-10)))
    new = (theta + alpha * x).float().double()                # set_param_values stores fp32
    ls0 = pol.n_params - pol.sizes[-1]
    new[ls0:] = torch.clamp(new[ls0:], min=pol.min_log_std)
    with torch.no_grad():
        out = dict(alpha=alpha, surr_before=float(adv_v.mean()), surr_after=float(surrogate(pol, new, theta, obs_v, act_v, adv_v)),
                   kl_dist=float(pol.mean_kl(new, theta, obs_v)), cg_iters_run=it, g=g, x=x)
    return new, out
