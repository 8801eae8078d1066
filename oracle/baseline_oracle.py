"""float64 restatement of mjrl's MLPBaseline (mjrl/mjrl/baselines/mlp_baseline.py:10-118) and of the minibatch loop it
fits with (mjrl/mjrl/utils/optimize_model.py: fit_data), the yardstick of amp_extensions_b200.baseline.

torch's own nn.Linear / ReLU / MSELoss and torch.optim.Adam(weight_decay) in float64 stand in for the reference's calls;
the permutation of each epoch is an input (np.random.permutation cannot be reproduced on the device).
"""
import numpy as np
import torch


def features(paths):
    """MLPBaseline._features for inp='obs': [clip(obs, -10, 10) / 10, (t/1000)^1..4] in float64 over the concatenated
    paths, t the step index within each path.  The matrix starts as np.ones and every column is overwritten: there is
    no constant column."""
    o = np.concatenate([p["observations"] for p in paths])
    o = np.clip(o, -10, 10) / 10.0
    if o.ndim > 2:
        o = o.reshape(o.shape[0], -1)
    N, n = o.shape
    feat_mat = np.ones((N, n + 4))
    feat_mat[:, :n] = o
    k = 0
    for p in paths:
        l = len(p["rewards"])
        al = np.arange(l) / 1000.0
        for j in range(4):
            feat_mat[k:k + l, -4 + j] = al ** (j + 1)
        k += l
    return feat_mat


def features_f32(paths):
    """The features as the reference's model sees them: cast to float32 once."""
    return features(paths).astype(np.float32)


def num_batches(n, batch_size):
    """fit_data's minibatch count: the `- 1` drops one full batch plus the remainder (zero below 2 * batch_size)."""
    return max(0, int(n // batch_size) - 1)


def make_model(sizes, params=None, dtype=torch.float64):
    """nn.Sequential(fc_0, relu_0, ..., fc_{L-1}) with widths `sizes`; params: flat vector in parameters() order."""
    model = torch.nn.Sequential()
    for i in range(len(sizes) - 1):
        model.add_module("fc_" + str(i), torch.nn.Linear(sizes[i], sizes[i + 1]))
        if i != len(sizes) - 2:
            model.add_module("relu_" + str(i), torch.nn.ReLU())
    model = model.to(dtype)
    if params is not None:
        set_flat(model, params)
    return model


def flat(model):
    return torch.cat([p.detach().reshape(-1) for p in model.parameters()])


def set_flat(model, v):
    v = torch.as_tensor(v)
    off = 0
    with torch.no_grad():
        for p in model.parameters():
            p.copy_(v[off:off + p.numel()].reshape(p.shape).to(p.dtype))
            off += p.numel()


def make_adam(model, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, exp_avg=None, exp_avg_sq=None, step=0):
    """torch.optim.Adam over the model, optionally continuing from a flat Adam state after `step` steps."""
    opt = torch.optim.Adam(model.parameters(), lr=lr, betas=betas, eps=eps, weight_decay=weight_decay)
    if exp_avg is not None:
        off = 0
        for p in model.parameters():
            k = p.numel()
            opt.state[p] = {"step": torch.tensor(float(step), dtype=torch.float64),
                            "exp_avg": torch.as_tensor(exp_avg[off:off + k]).reshape(p.shape).to(p.dtype).clone(),
                            "exp_avg_sq": torch.as_tensor(exp_avg_sq[off:off + k]).reshape(p.shape).to(p.dtype).clone()}
            off += k
    return opt


def predict(model, x):
    """model(features).ravel()"""
    with torch.no_grad():
        return model(torch.as_tensor(x).to(next(model.parameters()).dtype)).reshape(-1)


def minibatch_grads(model, x, y):
    """Gradients (parameters() order, flat) of MSELoss(mean) on one minibatch."""
    model.zero_grad()
    dt = next(model.parameters()).dtype
    loss = torch.nn.MSELoss()(model(torch.as_tensor(x).to(dt)), torch.as_tensor(y).to(dt).reshape(-1, 1))
    loss.backward()
    return torch.cat([p.grad.reshape(-1) for p in model.parameters()])


def fit(model, optimizer, x, y, perms, batch_size):
    """fit_data with the epochs' permutations given: for each, num_batches minibatches of disjoint rows, each an
    MSELoss(mean) backward and one optimizer step.  Returns the epochs' mean losses."""
    dt = next(model.parameters()).dtype
    x = torch.as_tensor(x).to(dt)
    y = torch.as_tensor(y).to(dt).reshape(-1, 1)
    loss_fn = torch.nn.MSELoss()
    out = []
    for perm in perms:
        perm = torch.as_tensor(perm, dtype=torch.int64)
        nb = num_batches(x.shape[0], batch_size)
        total = 0.0
        for mb in range(nb):
            idx = perm[mb * batch_size:(mb + 1) * batch_size]
            optimizer.zero_grad()
            loss = loss_fn(model(x[idx]), y[idx])
            loss.backward()
            optimizer.step()
            total += loss.item()
        out.append(total / nb if nb else float("nan"))
    return out


def error(model, x, y):
    """sum (y - y_hat)^2 / (sum y^2 + 1e-8) over all rows (MLPBaseline.fit's return_errors)."""
    y = torch.as_tensor(y).to(torch.float64).reshape(-1)
    e = y - predict(model, x).to(torch.float64)
    return float((e ** 2).sum() / ((y ** 2).sum() + 1e-8))
