"""How the library launches its kernels.  The host code (csrc/) launches every kernel through one function and sets a
kernel's dynamic shared-memory limit through one function that only ever raises it: the limit belongs to the kernel on
a device, so a handle that loads a smaller policy, NPG state or clip must not take shared memory away from another
handle's launches.  Every entry point that enqueues work checks the calling thread's device."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from tests import helpers as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "amp_extensions_b200", "csrc")
EINVAL = -1


def host_code():
    """{file: source without comments} of every source under csrc/."""
    out = {}
    for f in sorted(os.listdir(CSRC)):
        if f.endswith((".cu", ".cuh", ".inc", ".h")):
            with open(os.path.join(CSRC, f)) as fh:
                out[f] = re.sub(r"//[^\n]*|/\*.*?\*/", "", fh.read(), flags=re.S)
    return out


def test_every_launch_goes_through_one_function():
    code = host_code()
    assert [f for f, s in code.items() if "<<<" in s] == []
    calls = lambda name: [f for f, s in code.items() for _ in re.findall(r"\b" + name + r"\s*\(", s)]
    assert calls("cudaLaunchKernelEx") == ["launch.h"]
    assert calls("cudaFuncSetAttribute") == ["api.cu"]
    increments = [f for f, s in code.items() for _ in re.findall(r"g_launches\s*(?:\+\+|\+=|=)|\+\+\s*g_launches", s)]
    assert increments == ["launch.h"]


def test_precision_is_dispatched_in_one_place():
    """The only switch over SIMSTEP_PREC_* is with_elem's (launch.h)."""
    code = host_code()
    cases = [f for f, s in code.items() for _ in re.findall(r"\bcase\s+SIMSTEP_PREC_", s)]
    assert cases == ["launch.h"] * 3
    body = re.search(r"bool with_elem\(.*?\n\}", code["launch.h"], flags=re.S).group(0)
    assert len(re.findall(r"\bcase\s+SIMSTEP_PREC_", body)) == 3


# ---------------------------------------------------------------------------------------------------
# GPU: two handles on one device, the larger shape loaded first

def _engine():
    from amp_extensions_b200.engine import Engine
    return Engine(state_dim=8, action_dim=0, num_models=1, hidden_sizes=[], transform=False)


def _policy(sizes, seed):
    g = torch.Generator().manual_seed(seed)
    ws = [torch.randn(o, i, generator=g) / i ** 0.5 for i, o in zip(sizes[:-1], sizes[1:])]
    bs = [0.1 * torch.randn(o, generator=g) for o in sizes[1:]]
    log_std = -0.5 * torch.ones(sizes[-1])
    theta = torch.cat([t.reshape(-1) for w, b in zip(ws, bs) for t in (w, b)] + [log_std])  # mjrl's flat order
    return ws, bs, log_std, theta


def _load_policy(eng, sizes, seed):
    ws, bs, log_std, theta = _policy(sizes, seed)
    eng.load_policy(ws, bs, "tanh", log_std=log_std)
    eng.npg_init()
    eng.npg_params(theta.cuda())


def _rows(sizes, E, seed):
    g = torch.Generator().manual_seed(seed)
    obs = torch.randn(E, sizes[0], generator=g)
    act = torch.randn(E, sizes[-1], generator=g)
    adv = torch.randn(E, generator=g)
    return obs.cuda(), act.cuda(), adv.cuda()


BIG, SMALL = [226, 64, 64, 28], [8, 16, 4]  # policy_act needs 112000 and 19712 bytes of shared memory


@pytest.mark.gpu
def test_a_smaller_policy_on_another_handle_leaves_the_larger_one_running():
    """policy_act and npg_grad of handle A after handle B loaded a smaller policy and NPG state on the same device."""
    a, b = _engine(), _engine()
    _load_policy(a, BIG, 1)
    obs, act, adv = _rows(BIG, 1000, 2)
    noise = torch.randn(1000, BIG[-1], device="cuda")
    first = [t.clone() for t in a.policy_act(obs, noise)] + [a.npg_grad(obs, act, adv).clone()]
    _load_policy(b, SMALL, 3)
    obs_b, act_b, adv_b = _rows(SMALL, 100, 4)
    b.policy_act(obs_b)
    b.npg_grad(obs_b, act_b, adv_b)
    again = list(a.policy_act(obs, noise)) + [a.npg_grad(obs, act, adv)]
    torch.cuda.synchronize()
    for x, y in zip(again, first):
        assert torch.equal(x, y)


def _clip(n_frames):
    """The spinkick frames repeated until the clip has n_frames."""
    from amp_extensions_b200.character import humanoid3d
    from amp_extensions_b200.motion import MotionClip
    raw = H.spinkick_raw()
    raw = np.tile(raw, (-(-n_frames // raw.shape[0]), 1))[:n_frames]
    raw[:-1, 0] = raw[0, 0]  # every frame but the last has a duration (the spinkick's last frame has none)
    ch = humanoid3d()
    return ch, MotionClip.from_raw(raw, ch)


def _imitation_calls(eng, pose, vel, t, origin):
    reward, terms = eng.imitation_reward(pose, vel, t, origin, want_terms=True)
    return [reward.clone(), terms.clone()] + [x.clone() for x in eng.clip_sample(t, origin)]


@pytest.mark.gpu
@pytest.mark.parametrize("kernel, frames", [("generic", (234, 78)), ("h3d", (120, 78))])
def test_a_shorter_clip_on_another_handle_leaves_the_longer_one_running(monkeypatch, kernel, frames):
    """imitation_reward and clip_sample of handle A after handle B loaded a shorter clip on the same device.  Bytes of
    shared memory, A's then B's: generic reward 125472 and 71184, clip_sample 81440 and 27152; humanoid3d reward 219008
    and 204224, clip_sample 41760 and 27152."""
    monkeypatch.setenv("SIMSTEP_IMIT_GENERIC", "1" if kernel == "generic" else "0")
    a, b = _engine(), _engine()
    a.load_clip(*_clip(frames[0]))
    pose, vel, t, origin = (torch.from_numpy(x).float().cuda() for x in H.perturbed_poses(300, seed=5))
    first = _imitation_calls(a, pose, vel, t, origin)
    assert all(bool(x.isfinite().all()) for x in first)
    b.load_clip(*_clip(frames[1]))
    _imitation_calls(b, pose, vel, t, origin)
    again = _imitation_calls(a, pose, vel, t, origin)
    torch.cuda.synchronize()
    for x, y in zip(again, first):
        assert torch.equal(x, y)


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_enqueuing_from_another_device_is_refused():
    """A handle created on device 0, called from a thread whose current device is 1 with buffers on device 1."""
    eng = _engine()
    lib, h = eng.lib, eng._h
    p = lambda t: C.c_void_p(t.data_ptr())
    with torch.cuda.device(1):
        x = torch.ones(64, device="cuda:1")
        stats = torch.tensor([64.0, 64.0, 64.0], device="cuda:1", dtype=torch.float64)
        out = torch.empty(64, device="cuda:1")
        out2 = torch.empty(2, device="cuda:1", dtype=torch.float64)
        rcs = [lib.simstep_discount(h, p(x), None, None, None, None, 8, 8, C.c_float(0.9), C.c_float(1.0), p(out),
                                    None, None),
               lib.simstep_whiten(h, p(x), None, 64, p(stats), C.c_float(1e-8), p(out), None),
               lib.simstep_reduce_max_sum(h, p(x), 64, p(out2), None)]
        for rc in rcs:
            assert rc == EINVAL
            assert b"but the calling thread's current device is 1" in lib.simstep_last_error(h)
