"""On-device behaviour cloning of mjrl's Gaussian MLP policy (mjrl/mjrl/algos/behavior_cloning.py: BC), the warm start
MILO gives its policy before the first rollout (run.py:195-226) and run_BC.py on its own.

The parameters being fitted, their Adam state and the minibatch cursor live in the engine's handle (`simstep_bc_*`),
beside the policy the rollout samples from.  One optimiser step is four launches, so a whole epoch enqueues without a
host synchronisation (and can be captured in a CUDA graph).  The result is written in place into the engine's policy:
`Engine.generation` does not change, a DeviceRollout graph captured before keeps replaying with the cloned policy, and
an existing NPG state continues from the cloned parameters.

Deviation from the reference: `np.random.choice` cannot be reproduced on the device, so each epoch's minibatch rows are
drawn (with replacement, as np.random.choice draws them) from a seeded torch CUDA generator, or come from the caller as
an [epochs * int(n / batch_size), batch_size] int64 table (`idx=`).
"""
import time

import numpy as np
import torch

from . import parallel
from .npg import flat_params, set_flat_params

LOSS_TYPES = ("MSE", "MLE")


def _refuse_sharded():
    if parallel.world_size() > 1:
        raise RuntimeError("DeviceBC.fit: sequential minibatch Adam does not shard across ranks without changing its "
                           "result; fit on one rank")


def trainable_params(policy):
    """policy.trainable_params (the model's parameters, then log_std) when the object has it, else the same tensors
    from its FCNetwork layers and log_std."""
    if hasattr(policy, "trainable_params"):
        return list(policy.trainable_params)
    ts = []
    for l in policy.model.fc_layers:
        ts += [l.weight, l.bias]
    return ts + [policy.log_std]


def check_optimizer(opt):
    """The device step is torch.optim.Adam with one parameter group: refuse anything it would not reproduce."""
    if type(opt) is not torch.optim.Adam:
        raise NotImplementedError(f"BC on the device runs torch.optim.Adam, got {type(opt).__name__}")
    if len(opt.param_groups) != 1:
        raise NotImplementedError("BC on the device needs an optimiser with one parameter group")
    g = opt.param_groups[0]
    if g.get("amsgrad") or g.get("maximize") or g.get("decoupled_weight_decay"):
        raise NotImplementedError("amsgrad / maximize / decoupled weight decay Adam is not supported")


def statistics(obs, act):
    """BC.compute_transformations: per-column mean and population std (ddof 0) of the observations and actions, in
    float64 wherever the rows are."""
    obs, act = torch.as_tensor(obs).double(), torch.as_tensor(act).double()
    return obs.mean(0), obs.std(0, unbiased=False), act.mean(0), act.std(0, unbiased=False)


class BC:
    """The reference class's constructor and attributes (behavior_cloning.py): `policy`, `expert_paths`, `epochs`,
    `mb_size`, `loss_type`, `optimizer` (torch.optim.Adam over policy.trainable_params unless one is passed) and `log`
    (loss_before, epoch, loss_after, time after a fit).  set_transforms computes the expert statistics here on the
    host.  fit(data) / train() run on the GPU through DeviceBC."""

    def __init__(self, expert_paths, policy, epochs=5, batch_size=64, lr=1e-3, optimizer=None, loss_type='MSE',
                 set_transforms=False):
        if loss_type not in LOSS_TYPES:
            raise ValueError(f"loss_type must be 'MSE' or 'MLE', got {loss_type!r}")
        self.policy = policy
        self.expert_paths = expert_paths
        self.epochs = int(epochs)
        self.mb_size = int(batch_size)
        self.loss_type = loss_type
        self.min_log_std = float(getattr(policy, "min_log_std", -3.0))
        self.log = {}
        if set_transforms:
            self.apply_transformations(*self.compute_transformations())
        self.optimizer = torch.optim.Adam(trainable_params(policy), lr=lr) if optimizer is None else optimizer
        check_optimizer(self.optimizer)

    def _expert_rows(self):
        obs = np.concatenate([p["observations"] for p in self.expert_paths])
        act = np.concatenate([p["actions"] for p in self.expert_paths])
        return obs, act

    def compute_transformations(self):
        """(in_shift, in_scale, out_shift, out_scale) float64 numpy over the concatenated expert paths."""
        return tuple(t.numpy() for t in statistics(*self._expert_rows()))

    def apply_transformations(self, in_shift, in_scale, out_shift, out_scale):
        """set_transformations then set_variance_with_data, as the reference's constructor does."""
        self.set_transformations(in_shift, in_scale, out_shift, out_scale)
        self.set_variance_with_data(out_scale)

    def set_transformations(self, in_shift, in_scale, out_shift, out_scale):
        """Stored as float32 in policy.model (and old_model), through FCNetwork.set_transformations when it exists."""
        vals = [np.asarray(v, dtype=np.float64) for v in (in_shift, in_scale, out_shift, out_scale)]
        for model in (self.policy.model, getattr(self.policy, "old_model", None)):
            if model is None:
                continue
            if hasattr(model, "set_transformations"):
                model.set_transformations(*vals)
            else:
                model.in_shift, model.in_scale, model.out_shift, model.out_scale = (
                    torch.from_numpy(np.float32(v)) for v in vals)

    def set_variance_with_data(self, out_scale):
        """log_std = log(out_scale + 1e-12), written through set_param_values (which clamps at min_log_std)."""
        ls = np.log(np.asarray(out_scale, dtype=np.float64) + 1e-12)
        if hasattr(self.policy, "get_param_values") and hasattr(self.policy, "set_param_values"):
            params = self.policy.get_param_values()
            params[-ls.shape[0]:] = ls
            self.policy.set_param_values(params)
        else:
            theta = flat_params(self.policy).double()
            theta[-ls.shape[0]:] = torch.from_numpy(ls)
            set_flat_params(self.policy, theta, self.min_log_std)

    def fit(self, data, **kwargs):
        """BC.fit(data): data has 'observations' and 'expert_actions'; self.log gets loss_before, epoch, loss_after
        and time, and the policy object the fitted parameters."""
        if not all(k in data for k in ("observations", "expert_actions")):
            raise KeyError("data needs 'observations' and 'expert_actions'")
        ts = time.time()
        before, after = self._fit_rows(data["observations"], data["expert_actions"])
        self.log = {"loss_before": before, "epoch": self.epochs, "loss_after": after, "time": time.time() - ts}

    def train(self, **kwargs):
        """BC.train(): fit on the concatenated expert paths' observations and actions."""
        obs, act = self._expert_rows()
        self.fit(dict(observations=obs, expert_actions=act), **kwargs)

    def _fit_rows(self, obs, act):
        raise NotImplementedError("BC fits on the GPU: construct DeviceBC(engine_or_rollout, policy, ...)")


class DeviceBC(BC):
    """BC.fit on the GPU, written in place into the engine's policy.

        bc = DeviceBC(rollout, policy, expert_paths, epochs=5)   # rollout: DeviceRollout (or an Engine)
        bc.train()                                              # the reference's call: bc.log['loss_after'], ...
        before, after = bc.fit_tensors(obs, act, return_losses=True)   # device rows and scalars, no host copy
        bc.export()                                             # host policy and optimiser <- the device's
    """

    def __init__(self, rollout_or_engine, policy, expert_paths=None, epochs=5, batch_size=64, lr=1e-3, optimizer=None,
                 loss_type='MSE', set_transforms=False, seed=0):
        self.rollout = rollout_or_engine if hasattr(rollout_or_engine, "eng") else None
        self.eng = rollout_or_engine.eng if self.rollout is not None else rollout_or_engine
        super().__init__(expert_paths, policy, epochs, batch_size, lr, optimizer, loss_type, set_transforms=False)
        self.gen = torch.Generator(device=self.eng.device)
        self.gen.manual_seed(int(seed))
        if set_transforms:   # the statistics in float64 on the device, then the policy is uploaded again
            dev = self.eng.device
            obs, act = self._expert_rows()
            self.apply_transformations(*(t.cpu().numpy() for t in statistics(torch.as_tensor(obs).to(dev),
                                                                             torch.as_tensor(act).to(dev))))
            self._upload()
        elif not hasattr(self.eng, "policy_act_dim"):
            self._upload()
        self._attach()

    def _upload(self):
        if self.rollout is not None:
            self.rollout.load_policy(self.policy)
        else:
            from .rollout import _policy_parts
            ws, bs, name, (ish, isc, osh, osc), log_std = _policy_parts(self.policy)
            self.eng.load_policy(ws, bs, name, ish, isc, osh, osc, log_std)

    def _attach(self):
        """Create the device state from the host policy object's parameters and the optimiser's settings and state.
        Needed at construction and after a load_policy of the engine, which discards it."""
        opt = self.optimizer
        g = opt.param_groups[0]
        ps = trainable_params(self.policy)
        states = [opt.state.get(p, {}) for p in ps]
        have = ["exp_avg" in s for s in states[:-1]]
        if any(have) and not all(have):
            raise ValueError("the optimiser has state for some of the network's parameters only")
        m = v = None
        step = 0
        if all(have):
            def flat(key):
                return torch.cat([s[key].detach().float().reshape(-1).cpu() if key in s else torch.zeros(p.numel())
                                  for p, s in zip(ps, states)])
            m, v, step = flat("exp_avg"), flat("exp_avg_sq"), int(float(states[0]["step"]))
        self.n_params = self.eng.bc_init(self.mb_size, self.loss_type, flat_params(self.policy), lr=g["lr"],
                                         betas=g["betas"], eps=g["eps"], weight_decay=g["weight_decay"],
                                         min_log_std=self.min_log_std, exp_avg=m, exp_avg_sq=v, step=step)
        self._policy_gen = self.eng.policy_generation

    def _reattach(self):
        if self.eng.policy_generation != self._policy_gen:   # the policy was re-uploaded from the host object
            self._attach()

    def _rows(self, obs, act):
        dev = self.eng.device
        obs = torch.as_tensor(obs).to(dev, torch.float32)
        act = torch.as_tensor(act).to(dev, torch.float32)
        obs = obs.reshape(-1, self.eng.policy_obs_dim).contiguous()
        act = act.reshape(-1, self.eng.policy_act_dim).contiguous()
        if obs.shape[0] != act.shape[0]:
            raise ValueError(f"rows differ: observations {obs.shape[0]}, actions {act.shape[0]}")
        return obs, act

    def loss(self, obs, act):
        """The reference's loss over all rows (MSELoss(mean), or -mean log-likelihood) as a CUDA fp64 scalar; NaN
        for no rows."""
        self._reattach()
        obs, act = self._rows(obs, act)
        s = self.eng.bc_loss(obs, act)
        return s[1] / (s[0] * act.shape[1]) if self.loss_type == "MSE" else s[1] / s[0]

    def steps_per_epoch(self, n):
        """int(n / batch_size), the reference's minibatch count."""
        return int(n) // self.mb_size

    def fit_tensors(self, obs, act, idx=None, return_losses=False):
        """BC.fit on device rows: `epochs` epochs of int(n / batch_size) Adam steps, then the parameters are
        committed to the engine's policy (log_std clamped at min_log_std).  idx: the minibatch rows, int64
        [epochs * int(n / batch_size), batch_size]; default: drawn with replacement from the seeded generator.
        Returns (loss_before, loss_after) device scalars with return_losses."""
        _refuse_sharded()
        self._reattach()
        eng = self.eng
        obs, act = self._rows(obs, act)
        n = obs.shape[0]
        steps = self.steps_per_epoch(n)
        before = self.loss(obs, act) if return_losses else None
        if steps > 0 and self.epochs > 0:
            shape = (self.epochs * steps, self.mb_size)
            if idx is None:
                idx = torch.randint(0, n, shape, device=eng.device, generator=self.gen, dtype=torch.int64)
            else:
                idx = torch.as_tensor(idx).to(eng.device, torch.int64).reshape(shape)
                if bool((idx < 0).any()) or bool((idx >= n).any()):
                    raise ValueError(f"idx entries must lie in [0, {n})")
            for ep in range(self.epochs):
                eng.bc_fit(obs, act, idx[ep * steps:(ep + 1) * steps].reshape(-1).contiguous(), steps, restart=True)
        eng.bc_commit()
        if self.rollout is not None:   # what the next batches report as agent_infos['log_std']
            self.rollout.log_std = self.params()[-eng.policy_act_dim:]
        if return_losses:
            return before, self.loss(obs, act)
        return None

    def _fit_rows(self, obs, act):
        before, after = self.fit_tensors(obs, act, return_losses=True)
        self.export()
        return float(before), float(after)

    def params(self):
        """Current parameters (mjrl's flat order) as a CUDA fp32 tensor."""
        return self.eng.bc_read()["params"]

    def export(self):
        """Write the device parameters into the host policy object (through its own set_param_values when it has
        one, else into its tensors with the min_log_std clamp) and the Adam state into the optimiser.  MSE never
        trains log_std, so no optimiser state is written for it."""
        st = self.eng.bc_read()
        theta = st["params"].cpu()
        if hasattr(self.policy, "set_param_values"):
            self.policy.set_param_values(theta.numpy().copy(), set_new=True, set_old=True)
        else:
            set_flat_params(self.policy, theta, self.min_log_std)
        if st["step"] == 0:
            return theta
        ps = trainable_params(self.policy)
        off = 0
        for i, p in enumerate(ps):
            k = p.numel()
            if not (self.loss_type == "MSE" and i == len(ps) - 1):
                self.optimizer.state[p] = {
                    "step": torch.tensor(float(st["step"]), dtype=torch.float32),
                    "exp_avg": st["exp_avg"][off:off + k].reshape(p.shape).to(p.device, p.dtype),
                    "exp_avg_sq": st["exp_avg_sq"][off:off + k].reshape(p.shape).to(p.device, p.dtype)}
            off += k
        return theta
