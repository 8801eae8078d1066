"""On-device natural policy gradient step of mjrl's Gaussian MLP policy (mjrl/mjrl/algos/npg_cg.py: NPG.train_from_paths
with mjrl/mjrl/utils/cg_solve.py).

One `update` is: the vanilla gradient g = mean(adv * grad LL) over the rows, a conjugate-gradient solve of
(F + damping I) x = g with F the Hessian of MLP.mean_kl at new = old (its Fisher-vector products computed in closed form,
never as a matrix), the step theta += alpha x with alpha = sqrt(|delta / (g.x + 1e-10)|) (or a fixed learning rate),
the min_log_std clamp of set_param_values, and the diagnostics surr_after / kl_dist.  Every step is a libsimstep kernel on
the engine's stream; nothing waits for the host, so an update can be captured in a CUDA graph.  The new parameters are
written in place into the engine's policy: a DeviceRollout graph captured before keeps replaying with them.

Deviation from the reference: with hvp_sample_frac < 1 the Fisher rows are drawn with a seeded torch CUDA generator
(numpy's stream cannot be reproduced on the device), with replacement like np.random.choice.  Advantages are used as
given: whiten them first (RolloutBatch.normalize) where the reference's caller does.
"""
import numpy as np
import torch

from . import parallel


def flat_params(policy):
    """mjrl's get_param_values order: policy.trainable_params when the object has it, else every FCNetwork layer's
    weight and bias, then log_std (gaussian_mlp.py: trainable_params = list(model.parameters()) + [log_std])."""
    if hasattr(policy, "trainable_params"):
        ts = list(policy.trainable_params)
    else:
        ts = []
        for l in policy.model.fc_layers:
            ts += [l.weight, l.bias]
        ts.append(policy.log_std)
    return torch.cat([torch.as_tensor(np.asarray(t.data if hasattr(t, "data") else t, dtype=np.float32)).reshape(-1)
                      if not torch.is_tensor(t) else t.detach().float().reshape(-1).cpu() for t in ts])


def set_flat_params(policy, theta, min_log_std=None):
    """Writes theta (mjrl's flat order) into the policy object's tensors, clamping log_std like set_param_values."""
    theta = torch.as_tensor(theta).detach().float().cpu()
    if hasattr(policy, "trainable_params"):
        ts = list(policy.trainable_params)
    else:
        ts = []
        for l in policy.model.fc_layers:
            ts += [l.weight, l.bias]
        ts.append(policy.log_std)
    off = 0
    for i, t in enumerate(ts):
        n = t.numel()
        v = theta[off:off + n].reshape(t.shape).clone()
        if i == len(ts) - 1 and min_log_std is not None:
            v = torch.clamp(v, min=float(min_log_std))
        t.data = v.to(t.dtype)
        off += n
    if off != theta.numel():
        raise ValueError(f"parameter vector has {theta.numel()} entries, the policy {off}")


class DeviceNPG:
    """NPG policy step on the GPU.

        npg = DeviceNPG(rollout, policy)                # rollout: DeviceRollout (or an Engine with the policy loaded)
        adv = batch.normalize(batch.advantages(baseline, gamma, lam))
        stats = npg.update(batch, adv)                  # device scalars; the rollout's policy is updated in place
        npg.export_params()                             # host policy object <- the new parameters
    """

    def __init__(self, rollout_or_engine, policy, normalized_step_size=0.01, const_learn_rate=None, cg_iters=10,
                 damping=1e-4, hvp_sample_frac=1.0, seed=0):
        self.rollout = rollout_or_engine if hasattr(rollout_or_engine, "eng") else None
        self.eng = rollout_or_engine.eng if self.rollout is not None else rollout_or_engine
        self.policy = policy
        self.n_step_size = float(normalized_step_size)
        self.const_learn_rate = const_learn_rate
        self.cg_iters = int(cg_iters)
        self.damping = float(damping)
        self.hvp_sample_frac = float(hvp_sample_frac)
        self.min_log_std = float(getattr(policy, "min_log_std", -3.0))
        self.gen = torch.Generator(device=self.eng.device)
        self.gen.manual_seed(int(seed))
        if not hasattr(self.eng, "policy_act_dim"):   # no policy on the engine yet: upload the host object's
            if self.rollout is not None:
                self.rollout.load_policy(self.policy)
            else:
                from .rollout import _policy_parts
                ws, bs, name, (ish, isc, osh, osc), log_std = _policy_parts(self.policy)
                self.eng.load_policy(ws, bs, name, ish, isc, osh, osc, log_std)
        self._attach()

    def _attach(self):
        """Create the device NPG state with the host policy object's parameters.  Needed at construction and after a
        load_policy of the engine (which replaces the device parameters and discards the NPG state); other engine
        changes (cost, ensemble, termination) leave the policy and the NPG state alone."""
        self.n_params = self.eng.npg_init(self.min_log_std)
        theta = flat_params(self.policy)
        if theta.numel() != self.n_params:
            raise ValueError(f"policy has {theta.numel()} parameters, the engine's policy {self.n_params}")
        self.eng.npg_params(theta.to(self.eng.device))
        self._policy_gen = self.eng.policy_generation

    @staticmethod
    def _rows(x, width):
        return x.reshape(-1, width) if width else x.reshape(-1)

    def update(self, batch, advantages, valid=None):
        """One NPG step on the rows of `batch` (a RolloutBatch, or an (observations, actions) pair of device tensors)
        with per-row `advantages`; `valid` (uint8, same rows) masks rows out.  Returns device scalars: alpha, kl_dist,
        surr_before, surr_after, cg_iters_run.  With torch.distributed initialised every sum is all-reduced."""
        if self.eng.policy_generation != self._policy_gen:   # the policy was re-uploaded from the host object
            self._attach()
        eng = self.eng
        dev = eng.device
        obs, act = (batch.observations, batch.actions) if hasattr(batch, "observations") else batch
        # no copies for contiguous fp32 device tensors (rollout buffers); anything else is converted
        obs = torch.as_tensor(obs).to(dev, torch.float32).reshape(-1, obs.shape[-1]).contiguous()
        act = torch.as_tensor(act).to(dev, torch.float32).reshape(-1, act.shape[-1]).contiguous()
        adv = torch.as_tensor(advantages).to(dev, torch.float32).reshape(-1).contiguous()
        valid = None if valid is None else torch.as_tensor(valid).to(dev, torch.uint8).reshape(-1).contiguous()
        if act.shape[0] != obs.shape[0] or adv.shape[0] != obs.shape[0] or (valid is not None and valid.shape[0] != obs.shape[0]):
            raise ValueError(f"rows differ: obs {obs.shape[0]}, actions {act.shape[0]}, advantages {adv.shape[0]}"
                             + ("" if valid is None else f", valid {valid.shape[0]}"))
        n = obs.shape[0]
        idx = None
        if self.hvp_sample_frac < 1.0:
            k = max(1, int(self.hvp_sample_frac * n))
            idx = torch.randint(0, n, (k,), device=eng.device, generator=self.gen, dtype=torch.int64)
        g = parallel.all_reduce_sum(eng.npg_grad(obs, act, adv, valid))
        eng.npg_cg(eng.NPG_CG_START, g)
        eng.npg_prepare(obs, idx)
        for _ in range(self.cg_iters):
            z = parallel.all_reduce_sum(eng.npg_fvp(obs, valid, idx))
            eng.npg_cg(eng.NPG_CG_STEP, z, self.damping)
        if self.const_learn_rate is not None:
            eng.npg_apply(float(self.const_learn_rate), const_lr=True)
        else:
            eng.npg_apply(self.n_step_size)
        d = parallel.all_reduce_sum(eng.npg_diag(obs, act, adv, valid))
        sc = eng.npg_scalars()
        if self.rollout is not None:   # what the next batches report as agent_infos['log_std']
            self.rollout.log_std = eng.npg_params()[-eng.policy_act_dim:]
        rows = torch.clamp(d[0], min=1.0)
        return dict(alpha=sc[2], kl_dist=d[2] / rows, surr_before=sc[4], surr_after=d[1] / rows, cg_iters_run=sc[5])

    def params(self):
        """Current parameters (mjrl's flat order) as a CUDA fp32 tensor."""
        return self.eng.npg_params()

    def export_params(self):
        """Writes the device parameters into the host policy object in get_param_values order: through the object's
        own set_param_values when it has one (mjrl's MLP then also refreshes log_std_val and its old_* copies), else
        into its tensors with the min_log_std clamp."""
        theta = self.params().cpu()
        if hasattr(self.policy, "set_param_values"):
            self.policy.set_param_values(theta.numpy().copy(), set_new=True, set_old=True)
        else:
            set_flat_params(self.policy, theta, self.min_log_std)
        return theta

    def train_from_paths(self, paths):
        """The reference's call shape: concatenates observations / actions / advantages of the paths, uploads them and
        runs update()."""
        dev = self.eng.device
        obs = torch.from_numpy(np.concatenate([p["observations"] for p in paths]).astype(np.float32)).to(dev)
        act = torch.from_numpy(np.concatenate([p["actions"] for p in paths]).astype(np.float32)).to(dev)
        adv = torch.from_numpy(np.concatenate([p["advantages"] for p in paths]).astype(np.float32)).to(dev)
        return self.update((obs, act), adv)
