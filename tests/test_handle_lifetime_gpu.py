"""Lifetime of a handle's device state, through the raw C ABI: a failed load leaves its component unloaded instead of
half rewritten, a CUDA error is reported by the call that met it and by no later one, and destroying a handle returns
all of its device memory."""
import ctypes as C

import pytest
import torch

from tests import helpers as H

pytestmark = pytest.mark.gpu

EINVAL, ECUDA = -1, -2


def _engine(case, precision):
    from amp_extensions_b200.engine import Engine
    return Engine(case["S"], case["A"], case["N"], case["hidden"], dense_connect=case["dense"], activation=case["act"],
                  transform=True, precision=precision)


def _ensemble_args(case, null_member=None):
    """Pointer tables of simstep_load_ensemble; null_member: member whose layer-0 weight pointer is NULL."""
    nl = len(case["hidden"]) + 1
    keep = [t.float().contiguous() for t in case["tf"]]
    wp, bp = (C.c_void_p * (case["N"] * nl))(), (C.c_void_p * (case["N"] * nl))()
    for m in range(case["N"]):
        for l in range(nl):
            w, b = case["ws"][m][l].float().contiguous(), case["bs"][m][l].float().contiguous()
            keep += [w, b]
            wp[m * nl + l] = None if (m == null_member and l == 0) else w.data_ptr()
            bp[m * nl + l] = b.data_ptr()
    return wp, bp, (C.c_void_p * 6)(*[t.data_ptr() for t in keep[:6]]), keep


def _inputs(case, E=1000, seed=3):
    g = torch.Generator().manual_seed(seed)
    s = torch.randn(E, case["S"], generator=g).cuda()
    a = torch.randn(E, case["A"], generator=g).cuda()
    member = torch.randint(0, case["N"], (E,), generator=g, dtype=torch.int32).cuda()
    return s, a, member


def _step(eng, s, a, member):
    """(next_state, disc, done) of one simstep_step; the step counters start at zero for every call."""
    steps = torch.zeros(s.shape[0], dtype=torch.int32, device="cuda")
    out = eng.step(s, a, member, steps)
    torch.cuda.synchronize()
    return out


def _raw_step(eng, s, a, member):
    nxt = torch.empty_like(s)
    steps = torch.zeros(s.shape[0], dtype=torch.int32, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())
    return eng.lib.simstep_step(eng._h, p(s), p(a), p(member), p(steps), s.shape[0], p(nxt), None, None, None)


def _same(x, y):
    return all(torch.equal(u, v) for u, v in zip(x, y))


def test_failed_ensemble_reload_leaves_no_ensemble():
    case = H.tiny_case("tiny_dense")
    assert case["N"] >= 2
    s, a, member = _inputs(case)
    fresh = _engine(case, "fp16")
    fresh.load_ensemble(case["ws"], case["bs"], case["tf"])
    ref = _step(fresh, s, a, member)
    eng = _engine(case, "fp16")
    eng.load_ensemble(case["ws"], case["bs"], case["tf"])
    wp, bp, tp, keep = _ensemble_args(case, null_member=1)
    assert eng.lib.simstep_load_ensemble(eng._h, wp, bp, tp) == EINVAL
    # member 0 was rewritten before member 1 failed: the handle must not step on mixed weights
    assert _raw_step(eng, s, a, member) == EINVAL
    assert b"simstep_load_ensemble" in eng.lib.simstep_last_error(eng._h)
    wp, bp, tp, keep = _ensemble_args(case)
    assert eng.lib.simstep_load_ensemble(eng._h, wp, bp, tp) == 0
    assert _same(_step(eng, s, a, member), ref)
    eng.close()
    fresh.close()


def test_failed_train_init_is_reported_once_and_leaves_training_off():
    case = H.tiny_case("tiny_dense")
    s, a, member = _inputs(case)
    fresh = _engine(case, "tf32")
    fresh.load_ensemble(case["ws"], case["bs"], case["tf"])
    ref = _step(fresh, s, a, member)
    eng = _engine(case, "tf32")
    eng.load_ensemble(case["ws"], case["bs"], case["tf"])
    # the first training buffer alone is hundreds of GB: the allocation fails
    assert eng.lib.simstep_train_init(eng._h, 1 << 30, 0, 1e-4, 0.9, 0.999, 1e-8) == ECUDA
    assert _same(_step(eng, s, a, member), ref)
    # the failed init attached no training state (nor switched the handle to full-precision parameters)
    s3 = s[:256].reshape(1, 256, -1).expand(case["N"], -1, -1).contiguous()
    a3 = a[:256].reshape(1, 256, -1).expand(case["N"], -1, -1).contiguous()
    loss = torch.zeros(case["N"], dtype=torch.float64, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())
    assert eng.lib.simstep_train_step(eng._h, p(s3), p(a3), p(s3), 256, C.c_float(0.0), p(loss), None) == EINVAL
    eng.load_ensemble(case["ws"], case["bs"], case["tf"])
    assert _same(_step(eng, s, a, member), ref)
    eng.close()
    fresh.close()


def test_destroy_returns_every_component_s_device_memory():
    """One warm-up cycle (module loading, kernel attributes, torch's own buffers), then two cycles of a handle with
    every component loaded: the device's free memory after each equals its value after the warm-up."""
    from amp_extensions_b200.character import humanoid3d
    from amp_extensions_b200.motion import MotionClip
    case = H.tiny_case("tiny_dense")
    S, A = case["S"], case["A"]
    g = torch.Generator().manual_seed(5)
    rff_w, rff_b = torch.randn(256, S + A, generator=g), torch.rand(256, generator=g)
    sizes = [S, 32, A]
    pol_w = [torch.randn(o, i, generator=g) / i ** 0.5 for i, o in zip(sizes[:-1], sizes[1:])]
    pol_b = [torch.randn(o, generator=g) * 0.1 for o in sizes[1:]]
    ch = humanoid3d()
    clip = MotionClip.spinkick(ch)
    x = torch.randn(100_000, generator=g).cuda()
    torch.cuda.synchronize()

    def cycle():
        eng = _engine(case, "tf32")
        eng.load_ensemble(case["ws"], case["bs"], case["tf"])
        eng.load_rff(rff_w, rff_b, split=True, input_type="sa")
        eng.load_clip(ch, clip)
        eng.load_policy(pol_w, pol_b, "tanh", log_std=torch.full((A,), -0.5))
        eng.npg_init()
        eng.train_init(512)
        eng.moments(x)
        torch.cuda.synchronize()
        eng.close()
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        return torch.cuda.mem_get_info()[0]

    warm = cycle()
    assert [cycle(), cycle()] == [warm, warm]
