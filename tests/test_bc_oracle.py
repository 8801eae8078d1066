"""CPU checks of behaviour cloning's yardstick (oracle/bc_oracle.py) and host logic (amp_extensions_b200/bc.py): the
oracle's fit against a literal transcription of mjrl's BC.fit / mse_loss / mle_loss, the transformations and the
variance set from data by hand, the step count, and the refusals."""
import os
import socket
import sys
import tempfile

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import bc_oracle as bo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _FCNetwork(torch.nn.Module):
    """mjrl/mjrl/utils/fc_network.py in float64."""

    def __init__(self, sizes, nonlinearity):
        super().__init__()
        self.fc_layers = torch.nn.ModuleList([torch.nn.Linear(sizes[i], sizes[i + 1]).double()
                                              for i in range(len(sizes) - 1)])
        self.nonlinearity = torch.relu if nonlinearity == "relu" else torch.tanh
        self.set_transformations()

    def set_transformations(self, in_shift=None, in_scale=None, out_shift=None, out_scale=None):
        o, a = self.fc_layers[0].in_features, self.fc_layers[-1].out_features
        t = lambda v, d, fill: torch.from_numpy(np.float64(v)) if v is not None else torch.full((d,), fill, dtype=torch.float64)
        self.in_shift, self.in_scale = t(in_shift, o, 0.0), t(in_scale, o, 1.0)
        self.out_shift, self.out_scale = t(out_shift, a, 0.0), t(out_scale, a, 1.0)

    def forward(self, x):
        out = (x - self.in_shift) / (self.in_scale + 1e-8)
        for i in range(len(self.fc_layers) - 1):
            out = self.fc_layers[i](out)
            out = self.nonlinearity(out)
        out = self.fc_layers[-1](out)
        out = out * self.out_scale + self.out_shift
        return out


class _MLP:
    """mjrl/mjrl/policies/gaussian_mlp.py (the parts BC uses) in float64."""

    def __init__(self, sizes, nonlinearity, theta, min_log_std=-3.0):
        self.m = sizes[-1]
        self.min_log_std = min_log_std
        self.model = _FCNetwork(sizes, nonlinearity)
        self.log_std = torch.nn.Parameter(torch.zeros(self.m, dtype=torch.float64))
        self.trainable_params = list(self.model.parameters()) + [self.log_std]
        self.set_param_values(np.asarray(theta, dtype=np.float64))

    def get_param_values(self):
        return np.concatenate([p.contiguous().view(-1).data.numpy() for p in self.trainable_params])

    def set_param_values(self, new_params, set_new=True, set_old=True):
        cur = 0
        for p in self.trainable_params:
            k = p.numel()
            p.data = torch.from_numpy(new_params[cur:cur + k].reshape(p.shape)).double().clone()
            cur += k
        self.trainable_params[-1].data = torch.clamp(self.trainable_params[-1], self.min_log_std).data

    def new_dist_info(self, observations, actions):
        mean = self.model(observations)
        zs = (actions - mean) / torch.exp(self.log_std)
        LL = - 0.5 * torch.sum(zs ** 2, dim=1) + \
             - torch.sum(self.log_std) + \
             - 0.5 * self.m * np.log(2 * np.pi)
        return LL, mean, self.log_std


class _LiteralBC:
    """mjrl/mjrl/algos/behavior_cloning.py: BC.loss / mse_loss / mle_loss / fit, line by line, with
    np.random.choice replaced by the rows of `idx`."""

    def __init__(self, policy, epochs, batch_size, optimizer, loss_type):
        self.policy, self.epochs, self.mb_size, self.optimizer, self.loss_type = policy, epochs, batch_size, optimizer, loss_type
        self.loss_criterion = torch.nn.MSELoss()
        self.log = {}

    def loss(self, data, idx=None):
        return self.mle_loss(data, idx) if self.loss_type == 'MLE' else self.mse_loss(data, idx)

    def mle_loss(self, data, idx):
        idx = range(data['observations'].shape[0]) if idx is None else idx
        if type(data['observations']) == torch.Tensor:
            idx = torch.LongTensor(idx)
        obs = data['observations'][idx]
        act = data['expert_actions'][idx]
        LL, mu, log_std = self.policy.new_dist_info(obs, act)
        return -torch.mean(LL)

    def mse_loss(self, data, idx=None):
        idx = range(data['observations'].shape[0]) if idx is None else idx
        if type(data['observations']) is torch.Tensor:
            idx = torch.LongTensor(idx)
        obs = data['observations'][idx]
        act_expert = data['expert_actions'][idx]
        act_pi = self.policy.model(obs)
        return self.loss_criterion(act_pi, act_expert.detach())

    def fit(self, data, idx_table):
        num_samples = data["observations"].shape[0]
        self.log['loss_before'] = self.loss(data, idx=range(num_samples)).data.numpy().ravel()[0]
        k = 0
        for ep in range(self.epochs):
            for mb in range(int(num_samples / self.mb_size)):
                rand_idx = idx_table[k]
                k += 1
                self.optimizer.zero_grad()
                loss = self.loss(data, idx=rand_idx)
                loss.backward()
                self.optimizer.step()
        params_after_opt = self.policy.get_param_values()
        self.policy.set_param_values(params_after_opt, set_new=True, set_old=True)
        self.log['loss_after'] = self.loss(data, idx=range(num_samples)).data.numpy().ravel()[0]


@pytest.mark.parametrize("loss_type, sizes, act, n, bs, epochs, wd, tf", [
    ("MSE", (7, 16, 16, 3), "tanh", 300, 32, 2, 0.0, False),
    ("MLE", (7, 16, 16, 3), "tanh", 300, 32, 2, 0.0, True),
    ("MSE", (5, 8, 2), "relu", 130, 16, 3, 1e-2, True),
    ("MLE", (5, 8, 2), "relu", 130, 16, 1, 1e-2, False),
    ("MLE", (4, 1), "tanh", 64, 64, 3, 0.0, False),
    ("MSE", (11, 9, 6, 5, 4), "tanh", 200, 7, 1, 1e-3, True),
])
def test_oracle_fit_equals_a_literal_bc_fit(loss_type, sizes, act, n, bs, epochs, wd, tf):
    g = torch.Generator().manual_seed(n + bs)
    pol = bo.Policy(sizes, act, min_log_std=-1.2)
    theta = torch.randn(pol.n_params, generator=g, dtype=torch.float64) * 0.4
    theta[-sizes[-1]:] = -1.0 + 0.1 * torch.randn(sizes[-1], generator=g, dtype=torch.float64)
    obs = torch.randn(n, sizes[0], generator=g, dtype=torch.float64)
    act_ = torch.randn(n, sizes[-1], generator=g, dtype=torch.float64)
    steps = bo.step_count(n, bs)
    idx = torch.randint(0, n, (epochs * steps, bs), generator=g)
    idx[0, 1] = idx[0, 0]                                   # a row drawn twice counts twice
    lit_pol = _MLP(sizes, act, theta.numpy(), min_log_std=-1.2)
    if tf:
        shift = [torch.randn(d, generator=g, dtype=torch.float64).numpy() for d in (sizes[0], sizes[-1])]
        scale = [(0.5 + torch.rand(d, generator=g, dtype=torch.float64)).numpy() for d in (sizes[0], sizes[-1])]
        lit_pol.model.set_transformations(shift[0], scale[0], shift[1], scale[1])
        pol = bo.Policy(sizes, act, shift[0], scale[0], shift[1], scale[1], min_log_std=-1.2)
    lit = _LiteralBC(lit_pol, epochs, bs, torch.optim.Adam(lit_pol.trainable_params, lr=1e-2, weight_decay=wd),
                     loss_type)
    lit.fit(dict(observations=obs, expert_actions=act_), idx)
    params = bo.params_of(pol, theta)
    before, after = bo.fit(pol, params, bo.make_adam(params, loss_type, lr=1e-2, weight_decay=wd), obs, act_, idx,
                           epochs, bs, loss_type)
    assert torch.equal(bo.flat(params), torch.from_numpy(lit_pol.get_param_values()))
    assert before == lit.log['loss_before'] and after == lit.log['loss_after']
    if loss_type == "MSE":   # log_std never enters the graph: bit-identical, and the optimiser holds no state for it
        assert torch.equal(bo.flat(params)[-sizes[-1]:], theta[-sizes[-1]:])
        assert lit_pol.log_std not in lit.optimizer.state
    else:
        assert not torch.equal(bo.flat(params)[-sizes[-1]:], theta[-sizes[-1]:])


def test_commit_clamps_log_std_that_adam_drove_below_the_minimum():
    pol = bo.Policy((3, 2), "tanh", min_log_std=-0.6)
    theta = torch.zeros(pol.n_params, dtype=torch.float64)
    theta[-2:] = torch.tensor([-0.55, 0.3])
    g = torch.Generator().manual_seed(0)
    obs = torch.randn(256, 3, generator=g, dtype=torch.float64)
    act = 1e-3 * torch.randn(256, 2, generator=g, dtype=torch.float64)   # near-deterministic expert: std shrinks
    params = bo.params_of(pol, theta)
    opt = bo.make_adam(params, "MLE", lr=5e-2)
    idx = torch.randint(0, 256, (4 * 16, 16), generator=g)
    bo.fit(pol, params, opt, obs, act, idx, 4, 16, "MLE")
    ls = bo.flat(params)[-2:]
    assert float(ls[0]) == -0.6 and float(ls[1]) == -0.6


@pytest.mark.parametrize("n, bs, want", [(0, 64, 0), (63, 64, 0), (64, 64, 1), (127, 64, 1), (128, 64, 2),
                                         (1, 1, 1), (1023, 1024, 0), (100_000, 64, 1562), (1_000_000, 64, 15625)])
def test_step_count_is_int_n_over_batch(n, bs, want):
    from amp_extensions_b200.bc import DeviceBC
    assert bo.step_count(n, bs) == want
    d = object.__new__(DeviceBC)
    d.mb_size = bs
    assert d.steps_per_epoch(n) == want


class _HostPolicy:
    """The attributes of mjrl's MLP that the package reads, without get/set_param_values."""

    def __init__(self, sizes, min_log_std=-3.0):
        class M:
            pass
        self.model = M()
        self.model.fc_layers = [torch.nn.Linear(sizes[i], sizes[i + 1]) for i in range(len(sizes) - 1)]
        self.model.nonlinearity = torch.tanh
        self.log_std = torch.zeros(sizes[-1])
        self.min_log_std = min_log_std


def _paths():
    obs = np.array([[1.0, 2.0, -1.0], [3.0, 2.0, 0.0], [2.0, 2.0, 4.0], [6.0, 2.0, 1.0]])
    act = np.array([[0.5, 7.0], [-0.5, 7.0], [1.5, 7.0], [2.5, 7.0]])
    return [dict(observations=obs[:1], actions=act[:1]), dict(observations=obs[1:], actions=act[1:])]


def test_set_transforms_and_variance_by_hand():
    """Column 1 of the observations and column 1 of the actions are constant: std 0, in_scale 0 (the forward divides
    by 0 + 1e-8), and log(0 + 1e-12) = -27.6 clamped at min_log_std."""
    from amp_extensions_b200.bc import BC
    pol = _HostPolicy((3, 4, 2), min_log_std=-2.5)
    bc = BC(_paths(), pol, set_transforms=True)
    m = pol.model
    np.testing.assert_array_equal(m.in_shift.numpy(), np.float32([3.0, 2.0, 1.0]))
    np.testing.assert_array_equal(m.in_scale.numpy(), np.float32([np.sqrt(3.5), 0.0, np.sqrt(3.5)]))
    np.testing.assert_array_equal(m.out_shift.numpy(), np.float32([1.0, 7.0]))
    np.testing.assert_array_equal(m.out_scale.numpy(), np.float32([np.sqrt(1.25), 0.0]))
    assert m.in_shift.dtype == torch.float32
    np.testing.assert_array_equal(pol.log_std.numpy(), np.float32([np.log(np.sqrt(1.25) + 1e-12), -2.5]))
    np.testing.assert_array_equal(pol.log_std.numpy(), bo.variance_log_std([np.sqrt(1.25), 0.0], -2.5))
    for got, want in zip(bc.compute_transformations(), bo.transformations(*bc._expert_rows())):
        np.testing.assert_array_equal(got, want)
    # an mjrl-style object: through its own set_transformations and set_param_values (which clamps)
    mlp = _MLP((3, 4, 2), "tanh", np.zeros(3 * 4 + 4 + 4 * 2 + 2 + 2), min_log_std=-2.5)
    BC(_paths(), mlp, set_transforms=True)
    np.testing.assert_array_equal(mlp.model.in_shift.numpy(), [3.0, 2.0, 1.0])
    np.testing.assert_array_equal(mlp.log_std.data.numpy(), [np.log(np.sqrt(1.25) + 1e-12), -2.5])


def test_reference_constructor_and_refusals():
    from amp_extensions_b200.bc import BC
    pol = _HostPolicy((3, 4, 2))
    bc = BC(_paths(), pol, epochs=3, batch_size=2, lr=3e-3)
    assert bc.epochs == 3 and bc.mb_size == 2 and bc.loss_type == "MSE" and bc.log == {}
    assert type(bc.optimizer) is torch.optim.Adam and bc.optimizer.param_groups[0]["lr"] == 3e-3
    assert len(bc.optimizer.param_groups[0]["params"]) == 5 and bc.optimizer.param_groups[0]["params"][-1] is pol.log_std
    with pytest.raises(NotImplementedError, match="GPU"):
        bc.train()
    with pytest.raises(ValueError):
        BC(_paths(), pol, loss_type="L1")
    params = [l.weight for l in pol.model.fc_layers]
    for opt in (torch.optim.SGD(params, lr=0.1), torch.optim.AdamW(params), torch.optim.Adam(params, amsgrad=True),
                torch.optim.Adam(params, maximize=True)):
        with pytest.raises(NotImplementedError):
            BC(_paths(), pol, optimizer=opt)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from amp_extensions_b200.bc import DeviceBC
    bc = object.__new__(DeviceBC)  # the refusal comes before anything touches a device
    msgs = []
    for call in (lambda: bc.fit_tensors(None, None), lambda: bc.fit(dict(observations=None, expert_actions=None))):
        try:
            call()
            msgs.append(None)
        except RuntimeError as e:
            msgs.append(str(e))
    torch.save(msgs, os.path.join(out_dir, f"rank{rank}.pt"))
    dist.barrier()
    dist.destroy_process_group()


def test_fit_is_refused_under_torch_distributed():
    with tempfile.TemporaryDirectory() as d:
        mp.spawn(_worker, args=(2, _free_port(), d), nprocs=2, join=True)
        for r in range(2):
            msgs = torch.load(os.path.join(d, f"rank{r}.pt"))
            assert len(msgs) == 2 and all(m is not None and "does not shard" in m for m in msgs), msgs
