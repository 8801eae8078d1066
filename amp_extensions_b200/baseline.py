"""On-device MLP value baseline of mjrl (mjrl/mjrl/baselines/mlp_baseline.py: MLPBaseline, with the minibatch Adam loop
of mjrl/mjrl/utils/optimize_model.py: fit_data).

The network, its parameters and its Adam state live in the engine's handle (`simstep_baseline_*`).  Features are formed
inside the kernels from the observation rows and each row's step index within its path, so a T x E rollout batch is
predicted and fitted where it lies: nothing of it crosses to the host.  One optimiser step is four launches with the
minibatch cursor on the device, so a whole epoch enqueues without a host synchronisation (and can be captured in a CUDA
graph).

Deviation from the reference: `np.random.permutation` cannot be reproduced on the device, so each epoch's permutation
comes from a seeded torch CUDA generator, or from the caller (`perm=`).
"""
import numpy as np
import torch

from . import parallel


def time_index(done):
    """[T, E] int32 step index of every row within its path: a path starts at t = 0 and again after every done flag,
    exactly where RolloutBatch.segments() cuts the env columns."""
    T = done.shape[0]
    ar = torch.arange(T, device=done.device, dtype=torch.int64).reshape((T,) + (1,) * (done.dim() - 1)).expand(done.shape)
    start = torch.zeros(done.shape, device=done.device, dtype=torch.int64)
    start[1:] = torch.where(done[:-1].bool(), ar[1:], 0)
    return (ar - torch.cummax(start, dim=0).values).to(torch.int32)


def _refuse_sharded():
    if parallel.world_size() > 1:
        raise RuntimeError("DeviceMLPBaseline.fit: sequential minibatch Adam does not shard across ranks without "
                           "changing its result; fit on one rank (predict works per shard)")


class MLPBaseline:
    """The reference class's attributes on the host (mlp_baseline.py:10-36): `model` (nn.Sequential of fc_i Linear
    layers with ReLU between them, widths (n + 4,) + hidden_sizes + (1,)), `optimizer` (torch.optim.Adam with
    weight_decay = reg_coef), `batch_size`, `epochs`, `reg_coef`, `n`, `inp`.  Compute goes through DeviceMLPBaseline."""

    def __init__(self, env_spec, inp_dim=None, inp='obs', learn_rate=1e-3, reg_coef=0.0, batch_size=64, epochs=1,
                 use_gpu=False, hidden_sizes=(128, 128)):
        if inp != 'obs':
            raise NotImplementedError(f"MLPBaseline(inp={inp!r}): only inp='obs' is supported")
        self.n = inp_dim if inp_dim is not None else env_spec.observation_dim
        self.batch_size = batch_size
        self.epochs = epochs
        self.reg_coef = reg_coef
        self.use_gpu = use_gpu
        self.inp = inp
        self.hidden_sizes = hidden_sizes
        self.model = torch.nn.Sequential()
        sizes = (self.n + 4,) + tuple(hidden_sizes) + (1,)
        for i in range(len(sizes) - 1):
            self.model.add_module('fc_' + str(i), torch.nn.Linear(sizes[i], sizes[i + 1]))
            if i != len(sizes) - 2:
                self.model.add_module('relu_' + str(i), torch.nn.ReLU())
        self.optimizer = torch.optim.Adam(self.model.parameters(), lr=learn_rate, weight_decay=reg_coef)
        self.loss_function = torch.nn.MSELoss()


class DeviceMLPBaseline:
    """MLPBaseline.predict / fit on the GPU.

        vf = DeviceMLPBaseline(rollout, baseline)           # baseline: an object with MLPBaseline's attributes
        adv = batch.advantages(vf.predict_batch(batch), gamma, lam)
        err_before, err_after = vf.fit_batch(batch, batch.returns(gamma), return_errors=True)   # device scalars
        vf.export()                                         # host model and optimiser state <- the device's
    """

    def __init__(self, engine_or_rollout, baseline, seed=0):
        self.eng = engine_or_rollout.eng if hasattr(engine_or_rollout, "eng") else engine_or_rollout
        self.baseline = baseline
        if getattr(baseline, "inp", "obs") != "obs":
            raise NotImplementedError(f"MLPBaseline(inp={baseline.inp!r}): only inp='obs' is supported")
        self.layers = [m for m in baseline.model.modules() if isinstance(m, torch.nn.Linear)]
        self.sizes = [self.layers[0].in_features] + [l.out_features for l in self.layers]
        self.obs_dim = self.sizes[0] - 4
        self.batch_size = int(baseline.batch_size)
        self.epochs = int(baseline.epochs)
        self.gen = torch.Generator(device=self.eng.device)
        self.gen.manual_seed(int(seed))
        self._load()

    @classmethod
    def from_spec(cls, engine_or_rollout, env_spec, inp_dim=None, inp='obs', learn_rate=1e-3, reg_coef=0.0,
                  batch_size=64, epochs=1, use_gpu=False, hidden_sizes=(128, 128), seed=0):
        """The reference constructor's signature: builds the host MLPBaseline, then its device copy."""
        return cls(engine_or_rollout, MLPBaseline(env_spec, inp_dim, inp, learn_rate, reg_coef, batch_size, epochs,
                                                  use_gpu, hidden_sizes), seed=seed)

    def _params(self):
        return list(self.baseline.model.parameters())

    def _load(self):
        """Upload the host model's parameters and the optimiser's settings and state (a baseline already fitted on
        the host continues where it stopped)."""
        opt = self.baseline.optimizer
        if len(opt.param_groups) != 1:
            raise ValueError("the baseline's optimiser must have one parameter group")
        g = opt.param_groups[0]
        if g.get("amsgrad") or g.get("maximize"):
            raise NotImplementedError("amsgrad / maximize Adam is not supported")
        ps = self._params()
        flat = lambda ts: torch.cat([t.detach().float().reshape(-1).cpu() for t in ts])
        states = [opt.state.get(p, {}) for p in ps]
        have = all("exp_avg" in s for s in states)
        self.eng.baseline_init(self.sizes, self.batch_size, flat(ps), lr=g["lr"], betas=g["betas"], eps=g["eps"],
                               weight_decay=g["weight_decay"],
                               exp_avg=flat([s["exp_avg"] for s in states]) if have else None,
                               exp_avg_sq=flat([s["exp_avg_sq"] for s in states]) if have else None,
                               step=int(float(states[0]["step"])) if have else 0)

    def export(self):
        """Write the device parameters and Adam state into the host model and optimiser (checkpoints pickle them)."""
        st = self.eng.baseline_read()
        opt = self.baseline.optimizer
        off = 0
        for p in self._params():
            k = p.numel()
            with torch.no_grad():
                p.copy_(st["params"][off:off + k].reshape(p.shape).to(p.device, p.dtype))
            opt.state[p] = {"step": torch.tensor(float(st["step"]), dtype=torch.float32),
                            "exp_avg": st["exp_avg"][off:off + k].reshape(p.shape).to(p.device, p.dtype),
                            "exp_avg_sq": st["exp_avg_sq"][off:off + k].reshape(p.shape).to(p.device, p.dtype)}
            off += k

    # -- device API ------------------------------------------------------------------------------
    def _rows(self, batch):
        obs = batch.observations.reshape(-1, batch.observations.shape[-1])
        if obs.shape[1] != self.obs_dim:
            raise ValueError(f"observations have {obs.shape[1]} columns, the baseline expects {self.obs_dim}")
        return obs.contiguous(), time_index(batch.done).reshape(-1).contiguous()

    def predict_batch(self, batch):
        """Baseline values [T, E] of a RolloutBatch, time indices restarting after every done flag."""
        obs, t = self._rows(batch)
        return self.eng.baseline_predict(obs, t).reshape(batch.done.shape)

    def fit_batch(self, batch, returns, rows=None, return_errors=False, perm=None):
        """fit() on the rows of a RolloutBatch (all T * E, or the int64 flat row indices `rows`) against `returns`
        [T, E].  perm: one permutation of range(n) per epoch ([epochs, n], or [n] for one epoch); default: drawn
        from the seeded generator.  Returns (error_before, error_after) device scalars with return_errors."""
        _refuse_sharded()
        obs, t = self._rows(batch)
        y = returns.to(self.eng.device, torch.float32).reshape(-1).contiguous()
        return self._fit(obs, t, y, rows, return_errors, perm)

    def _error(self, obs, t, y, rows):
        pred = self.eng.baseline_predict(obs, t)
        if rows is not None:
            pred, y = pred[rows], y[rows]
        y = y.double()
        return ((y - pred.double()) ** 2).sum() / ((y ** 2).sum() + 1e-8)

    def _fit(self, obs, t, y, rows, return_errors, perm):
        dev = self.eng.device
        if rows is not None:
            rows = torch.as_tensor(rows).to(dev, torch.int64).reshape(-1)
        n = y.numel() if rows is None else rows.numel()
        if perm is not None:
            perm = torch.as_tensor(perm).to(dev, torch.int64).reshape(self.epochs, n)
        before = self._error(obs, t, y, rows) if return_errors else None
        n_steps = max(0, n // self.batch_size - 1)
        for ep in range(self.epochs):
            p = perm[ep] if perm is not None else torch.randperm(n, device=dev, generator=self.gen)
            idx = p if rows is None else rows[p]
            self.eng.baseline_fit(obs, t, y, idx.contiguous(), n_steps, restart=True)
        if return_errors:
            return before, self._error(obs, t, y, rows)
        return None

    # -- the reference's call shapes -------------------------------------------------------------
    def _path_rows(self, paths):
        dev = self.eng.device
        obs = np.concatenate([p["observations"] for p in paths]).reshape(-1, self.obs_dim)
        t = np.concatenate([np.arange(len(p["rewards"])) for p in paths])
        return (torch.from_numpy(obs.astype(np.float32)).to(dev).contiguous(),
                torch.from_numpy(t.astype(np.int32)).to(dev).contiguous())

    def predict(self, path):
        """MLPBaseline.predict(path): float32 numpy [len(path)]."""
        obs, t = self._path_rows([path])
        return self.eng.baseline_predict(obs, t).cpu().numpy()

    def fit(self, paths, return_errors=False):
        """MLPBaseline.fit(paths, return_errors): the paths' rows and returns are uploaded once; returns
        (error_before, error_after) as floats with return_errors."""
        _refuse_sharded()
        obs, t = self._path_rows(paths)
        y = torch.from_numpy(np.concatenate([p["returns"] for p in paths]).astype(np.float32)).to(self.eng.device)
        res = self._fit(obs, t, y.reshape(-1).contiguous(), None, return_errors, None)
        if return_errors:
            return float(res[0]), float(res[1])
        return None
