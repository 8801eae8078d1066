"""One MILO iteration on a B200 with the reference's objects swapped for amp_extensions_b200's (reference run.py:60-170
and mjrl/mjrl/algos/batch_reinforce.py:85-170, with the NPG update as an option):

  1. train the dynamics ensemble on an offline dataset            (run.py:80-93   -> DynamicsEnsemble.train)
  2. discrepancy threshold over the dataset                        (run.py:108     -> compute_threshold)
  3. IPM cost from expert (s, s') pairs                            (run.py:136-139 -> RBFLinearCost)
  4. roll the policy out in the learned-dynamics env               (sampler.py     -> DeviceRollout.collect)
  5. fit the cost on the rollout, recompute the rewards            (batch_reinforce.py:113-144)
  6. returns, GAE advantages, whitening, rollout statistics        (process_samples.py, batch_reinforce.py:135-141)
  7. with npg_steps > 0: that many rounds of collect -> advantages -> NPG policy step on the device (npg_cg.py,
     DeviceNPG.update)

Synthetic offline / expert data stand in for data/offline.pt and data/expert.pt (a download in the reference);
initial states come from the spin-kick clip without the simulator.  Run:  python examples/milo_iteration.py
"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


class GaussianMLP:
    """The attributes of mjrl's MLP policy that the rollout reads (gaussian_mlp.py:36-58)."""

    def __init__(self, obs_dim, act_dim, hidden=(32, 32), seed=0, init_log_std=-0.5):
        g = torch.Generator().manual_seed(seed)
        sizes = (obs_dim,) + tuple(hidden) + (act_dim,)

        class Net:
            pass

        self.model = Net()
        self.model.fc_layers = [torch.nn.Linear(sizes[i], sizes[i + 1]) for i in range(len(sizes) - 1)]
        for l in self.model.fc_layers:
            l.weight.data = torch.randn(l.weight.shape, generator=g) * (1.0 / l.weight.shape[1]) ** 0.5
            l.bias.data.zero_()
        self.model.fc_layers[-1].weight.data *= 1e-2
        self.model.nonlinearity = torch.tanh
        self.model.in_shift, self.model.in_scale = torch.zeros(obs_dim), torch.ones(obs_dim)
        self.model.out_shift, self.model.out_scale = torch.zeros(act_dim), torch.ones(act_dim)
        self.log_std = torch.full((act_dim,), float(init_log_std))


def main(num_envs=512, horizon=40, epochs=3, n_offline=4096, hidden=(128, 128), num_models=4, verbose=True, npg_steps=0):
    from amp_extensions_b200 import (AmpDataset, DynamicsEnsemble, ImitationReward, RBFLinearCost, VecSimEnv)
    from amp_extensions_b200.rollout import DeviceRollout
    S, A = 226, 28
    g = torch.Generator().manual_seed(0)
    imit = ImitationReward()
    # offline transitions around the reference motion: s ~ clip states, s' = s + small drift
    t = torch.rand(n_offline, generator=g) * float(imit.clip.duration)
    s = imit.reset_states(t.cuda()).cpu()
    a = torch.randn(n_offline, A, generator=g)
    s2 = s + 0.02 * torch.randn(n_offline, S, generator=g) + 0.01 * a.mean(dim=1, keepdim=True)
    ds = AmpDataset(s, a, s2)
    ens = DynamicsEnsemble(S, A, ds, None, num_models=num_models, batch_size=256, hidden_sizes=list(hidden),
                           dense_connect=True, transform=True, optim_args={"optim": "sgd", "lr": 0.02, "momentum": 0.9},
                           base_seed=100)
    fit = ens.train(epochs, grad_clip=1.0)                                            # 1
    ens.compute_threshold()                                                            # 2
    expert = torch.cat([s[:1024], s2[:1024]], dim=1)
    cost = RBFLinearCost(expert, feature_dim=512, input_type="ss", bw_quantile=0.1, lambda_b=0.0025, seed=100)   # 3
    env = VecSimEnv(ens, num_envs, horizon=horizon, reset_fn=VecSimEnv.clip_reset_fn(imit), reset_states=s[:1024], seed=1)
    env.reset()
    policy = GaussianMLP(S, A)
    ro = DeviceRollout(env, policy, seed=0)
    batch = ro.collect(horizon)                                                         # 4 (no cost yet: rewards 0)
    pi = torch.cat([batch.observations.reshape(-1, S), batch.next_observations.reshape(-1, S)], dim=1)
    mmd = cost.fit_cost(pi)                                                             # 5
    env.attach_cost(cost)
    env.reset()
    batch = ro.collect(horizon, graph=True)
    ret = batch.returns(0.995)                                                          # 6
    baseline = torch.zeros_like(ret)
    adv = batch.normalize(batch.advantages(baseline, 0.995, 0.97))
    stats = batch.statistics()
    paths = batch.paths(include_partial=False)
    out = dict(train_loss_first=[f[1] for f in fit], train_loss_best=[f[0] for f in fit], threshold=ens.threshold, mmd=mmd,
               env_steps=int(batch.rewards.numel()), trajectories=len(stats["ep_len"]), complete_paths=len(paths),
               mean_cost=stats["mean_cost"], adv_mean=float(adv.mean()), adv_std=float(adv.std(unbiased=False)),
               mean_return=float(ret[0].mean()), expert_cost=float(cost.get_expert_cost()))
    if npg_steps > 0:                                                                  # 7
        from amp_extensions_b200.npg import DeviceNPG
        npg = DeviceNPG(ro, policy)
        out["npg"] = []
        for _ in range(npg_steps):
            res = npg.update(batch, adv)
            out["npg"].append({k: float(v) for k, v in res.items()})
            env.reset()
            batch = ro.collect(horizon, graph=True)                                     # replays with the new policy
            ret = batch.returns(0.995)
            adv = batch.normalize(batch.advantages(torch.zeros_like(ret), 0.995, 0.97))
        npg.export_params()
    if verbose:
        for k, v in out.items():
            print(f"{k:18s} {v}")
    return out, batch


if __name__ == "__main__":
    main()
