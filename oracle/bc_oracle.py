"""float64 restatement of mjrl's behaviour cloning (mjrl/mjrl/algos/behavior_cloning.py: BC.fit, mse_loss, mle_loss,
compute_transformations, set_variance_with_data) on the Gaussian MLP policy (mjrl/mjrl/policies/gaussian_mlp.py over
mjrl/mjrl/utils/fc_network.py:42-55), the yardstick of amp_extensions_b200.bc.  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

torch's own F.linear, MSELoss and torch.optim.Adam in float64 stand in for the reference's calls.  The parameters are
separate leaf tensors in get_param_values order (per layer W [out][in], b [out], then log_std), so that in MSE mode
log_std has no gradient and Adam never touches it, as in the reference.  np.random.choice is replaced by an index table
[epochs * int(n / B), B] (rows drawn with replacement).
"""
import numpy as np
import torch
import torch.nn.functional as F

from oracle.npg_oracle import Policy  # noqa: F401  (shapes and transformations of a policy)


def step_count(n, batch_size):
    """BC.fit's minibatches per epoch: int(n / batch_size), with no `- 1` (fit_data's rule for the baseline has one)."""
    return int(n / batch_size)


def params_of(pol, theta):
    """Leaf float64 tensors [W_0, b_0, ..., W_L, b_L, log_std] of a flat vector."""
    ws, bs, ls = pol.unflatten(torch.as_tensor(theta, dtype=torch.float64))
    out = []
    for w, b in zip(ws, bs):
        out += [w.clone(), b.clone()]
    out.append(ls.clone())
    return [p.requires_grad_(True) for p in out]


def flat(params):
    return torch.cat([p.detach().reshape(-1) for p in params])


def mean(pol, params, obs):
    """FCNetwork.forward: x = (obs - in_shift) / (in_scale + 1e-8), act(fc) layers, out * out_scale + out_shift."""
    act = torch.relu if pol.nonlinearity == "relu" else torch.tanh
    x = (torch.as_tensor(obs, dtype=torch.float64) - pol.in_shift) / (pol.in_scale + 1e-8)
    L = (len(params) - 1) // 2
    for l in range(L - 1):
        x = act(F.linear(x, params[2 * l], params[2 * l + 1]))
    x = F.linear(x, params[2 * L - 2], params[2 * L - 1])
    return x * pol.out_scale + pol.out_shift


def mse_loss(pol, params, obs, act):
    return torch.nn.MSELoss()(mean(pol, params, obs), torch.as_tensor(act, dtype=torch.float64))


def mle_loss(pol, params, obs, act):
    """-mean(LL), LL = -1/2 sum z^2 - sum log_std - m/2 log 2 pi with z = (a - mu) / exp(log_std)."""
    mu = mean(pol, params, obs)
    log_std = params[-1]
    zs = (torch.as_tensor(act, dtype=torch.float64) - mu) / torch.exp(log_std)
    LL = -0.5 * torch.sum(zs ** 2, dim=1) + -torch.sum(log_std) + -0.5 * mu.shape[1] * np.log(2 * np.pi)
    return -torch.mean(LL)


def loss(loss_type, pol, params, obs, act):
    return (mse_loss if loss_type == "MSE" else mle_loss)(pol, params, obs, act)


def make_adam(params, loss_type, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, exp_avg=None,
              exp_avg_sq=None, step=0):
    """torch.optim.Adam over the parameters, optionally continuing from flat moments after `step` steps (MSE: no state
    for log_std, which the reference never steps)."""
    opt = torch.optim.Adam(params, lr=lr, betas=betas, eps=eps, weight_decay=weight_decay)
    if exp_avg is not None and step > 0:
        off = 0
        for i, p in enumerate(params):
            k = p.numel()
            if not (loss_type == "MSE" and i == len(params) - 1):
                opt.state[p] = {"step": torch.tensor(float(step), dtype=torch.float64),
                                "exp_avg": torch.as_tensor(exp_avg[off:off + k]).reshape(p.shape).double().clone(),
                                "exp_avg_sq": torch.as_tensor(exp_avg_sq[off:off + k]).reshape(p.shape).double().clone()}
            off += k
    return opt


def minibatch_grads(loss_type, pol, theta, obs, act, rows):
    """Flat gradient of one minibatch's loss (log_std's is 0 in MSE mode, where it is not in the graph)."""
    params = params_of(pol, theta)
    rows = torch.as_tensor(rows, dtype=torch.int64)
    obs, act = torch.as_tensor(obs, dtype=torch.float64), torch.as_tensor(act, dtype=torch.float64)
    loss(loss_type, pol, params, obs[rows], act[rows]).backward()
    return torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1) for p in params])


def commit(pol, params):
    """set_param_values(get_param_values(), set_new=True, set_old=True): log_std clamped at min_log_std."""
    with torch.no_grad():
        params[-1].data = torch.clamp(params[-1], pol.min_log_std).data


def fit(pol, params, optimizer, obs, act, idx, epochs, batch_size, loss_type):
    """BC.fit with np.random.choice replaced by the rows of `idx` ([epochs * int(n / B), B]); the parameters are
    updated in place and committed.  Returns (loss_before, loss_after) as floats."""
    obs, act = torch.as_tensor(obs, dtype=torch.float64), torch.as_tensor(act, dtype=torch.float64)
    n = obs.shape[0]
    with torch.no_grad():
        before = float(loss(loss_type, pol, params, obs, act))
    steps = step_count(n, batch_size)
    idx = torch.as_tensor(idx, dtype=torch.int64).reshape(-1, batch_size) if steps else None
    for ep in range(epochs):
        for mb in range(steps):
            rows = idx[ep * steps + mb]
            optimizer.zero_grad()
            lo = loss(loss_type, pol, params, obs[rows], act[rows])
            lo.backward()
            optimizer.step()
    commit(pol, params)
    with torch.no_grad():
        after = float(loss(loss_type, pol, params, obs, act))
    return before, after


def transformations(obs, act):
    """BC.compute_transformations in float64: (in_shift, in_scale, out_shift, out_scale), population std."""
    obs, act = np.asarray(obs, dtype=np.float64), np.asarray(act, dtype=np.float64)
    return np.mean(obs, axis=0), np.std(obs, axis=0), np.mean(act, axis=0), np.std(act, axis=0)


def variance_log_std(out_scale, min_log_std):
    """set_variance_with_data: float32(log(out_scale + 1e-12)) clamped at min_log_std (set_param_values)."""
    return np.maximum(np.float32(np.log(np.asarray(out_scale, dtype=np.float64) + 1e-12)), np.float32(min_log_std))

