"""CPU checks of the MLP value baseline's yardstick (oracle/baseline_oracle.py) and host logic
(amp_extensions_b200/baseline.py): the reference's features and minibatch count, the oracle's fit against a literal
transcription of mjrl's fit_data, the time index against RolloutBatch.segments(), and the refusals."""
import os
import socket
import sys
import tempfile

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import baseline_oracle as bo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _path(obs):
    return {"observations": np.asarray(obs, dtype=np.float64), "rewards": np.zeros(len(obs))}


def test_features_clip_scale_and_time_columns_by_hand():
    obs = np.array([[0.5, -12.0, 10.0], [25.0, -10.0, -3.0], [0.0, 1e-3, 7.25]])
    f = bo.features([_path(obs[:2]), _path(obs[2:])])
    assert f.shape == (3, 7) and f.dtype == np.float64
    np.testing.assert_array_equal(f[:, :3], [[0.05, -1.0, 1.0], [1.0, -1.0, -0.3], [0.0, 1e-4, 0.725]])
    # t restarts in every path: rows 0 and 2 are t = 0 (all four powers 0, no constant column of ones), row 1 is t = 1
    np.testing.assert_array_equal(f[0, 3:], [0, 0, 0, 0])
    np.testing.assert_array_equal(f[2, 3:], [0, 0, 0, 0])
    np.testing.assert_allclose(f[1, 3:], [1e-3, 1e-6, 1e-9, 1e-12], rtol=1e-15)
    long = bo.features([_path(np.zeros((1500, 1)))])
    np.testing.assert_allclose(long[1234, 1:], [1.234, 1.234 ** 2, 1.234 ** 3, 1.234 ** 4], rtol=1e-15)
    assert bo.features_f32([_path(obs)]).dtype == np.float32


@pytest.mark.parametrize("n, bs, want", [(0, 64, 0), (63, 64, 0), (64, 64, 0), (127, 64, 0), (128, 64, 1),
                                         (129, 64, 1), (6144, 64, 95), (1, 1, 0), (2, 1, 1), (63, 1, 62),
                                         (1_280_000, 64, 19_999), (511, 256, 0), (512, 256, 1)])
def test_step_count_is_n_over_batch_minus_one(n, bs, want):
    assert bo.num_batches(n, bs) == want


def _literal_fit_data(model, x, y, optimizer, loss_func, batch_size, epochs, perms):
    """mjrl/mjrl/utils/optimize_model.py: fit_data, line by line, with np.random.permutation replaced by `perms`."""
    num_samples = x.shape[0]
    epoch_losses = []
    for ep in range(epochs):
        rand_idx = torch.LongTensor(perms[ep])
        ep_loss = 0.0
        num_batches = int(num_samples // batch_size) - 1
        for mb in range(num_batches):
            data_idx = rand_idx[mb * batch_size:(mb + 1) * batch_size]
            batch_x = x[data_idx]
            batch_y = y[data_idx]
            optimizer.zero_grad()
            yhat = model(batch_x)
            loss = loss_func(yhat, batch_y)
            loss.backward()
            optimizer.step()
            ep_loss += loss.to('cpu').data.numpy().ravel()[0]
        epoch_losses.append(ep_loss * 1.0 / num_batches)
    return epoch_losses


@pytest.mark.parametrize("sizes, n, bs, epochs, wd", [((9, 16, 16, 1), 300, 32, 2, 0.0), ((5, 1), 200, 16, 1, 1e-2),
                                                      ((21, 8, 4, 2, 1), 333, 64, 3, 1e-3)])
def test_oracle_fit_equals_a_literal_fit_data(sizes, n, bs, epochs, wd):
    g = torch.Generator().manual_seed(n)
    x = torch.randn(n, sizes[0], generator=g, dtype=torch.float64)
    y = torch.randn(n, 1, generator=g, dtype=torch.float64)
    perms = [torch.randperm(n, generator=g).numpy() for _ in range(epochs)]
    torch.manual_seed(3)
    a = bo.make_model(sizes)
    b = bo.make_model(sizes, bo.flat(a))
    lit = _literal_fit_data(a, x, y, torch.optim.Adam(a.parameters(), lr=1e-2, weight_decay=wd), torch.nn.MSELoss(),
                            bs, epochs, perms)
    got = bo.fit(b, bo.make_adam(b, lr=1e-2, weight_decay=wd), x, y, perms, bs)
    assert torch.equal(bo.flat(a), bo.flat(b))
    np.testing.assert_array_equal(np.float64(lit), got)


def test_oracle_adam_continues_from_an_imported_state():
    """Two fits in a row equal a first fit plus a fresh model and optimiser built from its exported state."""
    g = torch.Generator().manual_seed(1)
    x = torch.randn(200, 6, generator=g, dtype=torch.float64)
    y = torch.randn(200, generator=g, dtype=torch.float64)
    perms = [torch.randperm(200, generator=g) for _ in range(2)]
    torch.manual_seed(0)
    a = bo.make_model((6, 8, 1))
    opt = bo.make_adam(a, lr=1e-2, weight_decay=1e-3)
    bo.fit(a, opt, x, y, perms[:1], 32)
    st = [opt.state[p] for p in a.parameters()]
    b = bo.make_model((6, 8, 1), bo.flat(a))
    opt_b = bo.make_adam(b, lr=1e-2, weight_decay=1e-3, exp_avg=torch.cat([s["exp_avg"].reshape(-1) for s in st]),
                         exp_avg_sq=torch.cat([s["exp_avg_sq"].reshape(-1) for s in st]), step=int(st[0]["step"]))
    bo.fit(a, opt, x, y, perms[1:], 32)
    bo.fit(b, opt_b, x, y, perms[1:], 32)
    assert torch.equal(bo.flat(a), bo.flat(b))


class _Batch:
    """The parts of RolloutBatch that segments() reads."""

    def __init__(self, done):
        self.done = done
        self.T, self.E = done.shape

    segments = __import__("amp_extensions_b200.rollout", fromlist=["RolloutBatch"]).RolloutBatch.segments


@pytest.mark.parametrize("T, E, p", [(1, 5, 0.3), (32, 64, 0.1), (7, 33, 0.5), (40, 16, 0.0), (50, 9, 0.02)])
def test_time_index_restarts_where_segments_cut(T, E, p):
    from amp_extensions_b200.baseline import time_index
    g = torch.Generator().manual_seed(T * 1000 + E)
    done = (torch.rand(T, E, generator=g) < p).to(torch.uint8)
    done[:, 0] = 0                    # a column with no done at all
    if T > 3:
        done[T - 1, 1] = 1            # a column whose path ends at the last step
        done[0, 2] = 1                # a path that ends at the first step
    t = time_index(done)
    assert t.dtype == torch.int32 and t.shape == (T, E)
    want = torch.full((T, E), -1, dtype=torch.int32)
    for e, t0, t1, _ in _Batch(done).segments():
        want[t0:t1, e] = torch.arange(t1 - t0, dtype=torch.int32)
    assert torch.equal(t, want)


def test_env_features_input_is_refused():
    from amp_extensions_b200.baseline import MLPBaseline

    class Spec:
        observation_dim = 7

    with pytest.raises(NotImplementedError):
        MLPBaseline(Spec(), inp='env_features')
    b = MLPBaseline(Spec(), hidden_sizes=(5,), reg_coef=0.25)
    names = [n for n, _ in b.model.named_children()]
    assert names == ["fc_0", "relu_0", "fc_1"] and b.model.fc_0.in_features == 11
    assert b.optimizer.param_groups[0]["weight_decay"] == 0.25


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from amp_extensions_b200.baseline import DeviceMLPBaseline
    vf = object.__new__(DeviceMLPBaseline)  # the refusal comes before anything touches a device
    msgs = []
    for call in (lambda: vf.fit([], return_errors=True), lambda: vf.fit_batch(None, None)):
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
