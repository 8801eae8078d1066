"""CPU: the oracle restatement against the golden vectors produced by the reference's own code."""
import os

import numpy as np
import pytest
import torch

from oracle import milo_oracle as mo
from tests import helpers as H

GOLDEN_THREADS = 8


@pytest.fixture(autouse=True, scope="module")
def golden_thread_count():
    """The float32 golden vectors were written with GOLDEN_THREADS torch intra-op threads.  The CPU GEMM (MKL) splits
    its sums by thread count, so the same ops reproduce the stored bits only with that count, whatever the host's
    number of cores.  The bits also depend on the MKL build and on the instruction set its kernels use (they are
    reproduced by the MKL that torch 2.11 ships, on AVX-512); pinning the thread count removes only the core-count
    dependence."""
    before = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(before)


@pytest.mark.parametrize("tag", ["tiny_dense", "tiny_plain_tanh"])
def test_forward_and_discrepancy_match_reference(tag):
    c = H.tiny_case(tag)
    preds = mo.ensemble_forward(c["ws"], c["bs"], c["tf"], c["xs"], c["xa"], c["dense"], c["act"])
    assert torch.equal(preds, c["preds"])  # same ops, same order: bit-exact
    pn = torch.stack([mo.dynamics_forward(w, b, c["tf"], c["xs"], c["xa"], c["dense"], c["act"], unnormalize_out=False)
                      for w, b in zip(c["ws"], c["bs"])])
    assert torch.equal(pn, c["preds_norm"])
    assert torch.equal(mo.discrepancy_from_preds(preds), c["disc"])


@pytest.mark.parametrize("tag", ["tiny_dense", "tiny_plain_tanh"])
def test_transformations_and_threshold_match_reference(tag):
    c = H.tiny_case(tag)
    tf = mo.get_transformations(*c["ds"])
    for a, b in zip(tf, c["tf"]):
        assert torch.equal(a, b)
    thr = mo.compute_threshold(c["ws"], c["bs"], c["tf"], c["ds"][0], c["ds"][1], 256, c["dense"]) \
        if c["act"] == "relu" else None
    if thr is not None:
        assert thr == pytest.approx(c["threshold"], rel=1e-6)


def test_layer_shapes_of_north_star_config():
    fan_in, fan_out = mo.layer_input_sizes(254, 226, [512] * 4, True)
    assert fan_in == [254, 766, 1278, 1790, 2302]  # SURVEY.md section 0, dynamics.py:412-420
    assert fan_out == [512, 512, 512, 512, 226]
    fan_in, _ = mo.layer_input_sizes(254, 226, [1024] * 4, True)
    assert fan_in == [254, 1278, 2302, 3326, 4350]


def test_north_star_init_is_the_reference_init():
    c = H.ns_case()
    for k in range(c["N"]):
        flat = [x for pair in zip(c["ws"][k], c["bs"][k]) for x in pair]
        np.testing.assert_allclose([float(v.double().sum()) for v in flat], c["wsum"][k], rtol=0, atol=1e-9)
        np.testing.assert_allclose([float(v.double().abs().sum()) for v in flat], c["wabs"][k], rtol=1e-12)


def test_north_star_forward_matches_reference():
    c = H.ns_case()
    preds = mo.ensemble_forward(c["ws"], c["bs"], c["tf"], c["xs"], c["xa"])
    assert torch.equal(preds, c["preds"])
    assert torch.equal(mo.discrepancy_from_preds(preds), c["disc"])
    s, a, _ = H.synth_dataset(8192, 226, 28, 0)
    n = c["threshold_rows"]
    assert mo.compute_threshold(c["ws"], c["bs"], c["tf"], s[:n], a[:n]) == pytest.approx(c["threshold"], rel=1e-6)


@pytest.mark.parametrize("tag,D", [("cost64", 64), ("cost512", 512)])
def test_rff_cost_matches_reference(tag, D):
    g = H.golden()
    c = H.ns_case()
    expert = H.ns_expert()
    if tag == "cost64":
        assert torch.equal(expert, H.t(g["cost64/expert"]))
    cost = mo.RffCostOracle(expert, feature_dim=D, input_type="ss", bw_quantile=0.1, lambda_b=0.0025, seed=100)
    assert cost.bw == pytest.approx(float(g[f"{tag}/bw"]), rel=0, abs=0)
    if D == 64:
        assert torch.equal(cost.rff_weight, H.t(g["cost64/rff_w"]))
        assert torch.equal(cost.rff_bias, H.t(g["cost64/rff_b"]))
    assert torch.equal(cost.phi_e, H.t(g[f"{tag}/phi_e"]))
    nxt = H.t(g[f"{tag}/next"])
    pi = torch.cat([c["xs"], nxt], dim=1)
    assert torch.equal(cost.get_rep(pi), H.t(g[f"{tag}/rep"]))
    assert cost.fit_cost(pi) == pytest.approx(float(g[f"{tag}/mmd"]), rel=1e-7)
    assert torch.equal(cost.w, H.t(g[f"{tag}/w"]))
    assert torch.equal(cost.get_costs(pi), H.t(g[f"{tag}/costs"]))
    assert float(cost.get_expert_cost()) == pytest.approx(float(g[f"{tag}/expert_cost"]), rel=1e-7)
    total, info = cost.get_bonus_costs(c["xs"], c["xa"], c["disc"], c["threshold"], next_states=nxt)
    assert torch.equal(total, H.t(g[f"{tag}/total"]))
    for k in ("bonus", "ipm", "v_targ", "cost"):
        assert torch.equal(info[k], H.t(g[f"{tag}/info_{k}"]))


# ---- SimEnv restatement: no reference vectors exist (gym + SWIG simulator), hand-built known answers ----

def _standing_state():
    s = np.zeros((1, 226))
    s[0, 0] = 0.9          # root height
    for b in range(15):
        s[0, 9 * b + 5] = 1.0  # normals point up
    return s


def test_simenv_no_collision_when_standing():
    s = _standing_state()
    assert not mo.simenv_collided(s)[0]


def test_simenv_sphere_threshold_is_radius_plus_1e_4():
    # neck (body 2, diameter 0.205): world y = s[0] + s[9*2+2]; sim_env.py:188-189
    for dy, want in ((0.1025 + 0.0001 + 1e-6, False), (0.1025 + 0.0001 - 1e-6, True)):
        s = _standing_state()
        s[0, 9 * 2 + 2] = dy - s[0, 0]
        assert bool(mo.simenv_collided(s)[0]) is want


def test_simenv_capsule_uses_both_end_caps():
    # right knee (body 4: diameter .10, height .31): centre at y=0.2, tilted so that one cap reaches the ground
    s = _standing_state()
    s[0, 9 * 4 + 2] = 0.2 - s[0, 0]
    s[0, 9 * 4 + 5] = 0.5
    assert not mo.simenv_collided(s)[0]           # 0.2 - 0.155*0.5 = 0.1225 > 0.0501
    s[0, 9 * 4 + 5] = -1.0
    assert mo.simenv_collided(s)[0]               # 0.2 - 0.155 = 0.045 <= 0.0501 (top cap, normal flipped)
    # ankles (bodies 5, 11) are boxes and never count (sim_env.py:238-244)
    s = _standing_state()
    s[0, 9 * 5 + 2] = -5.0
    assert not mo.simenv_collided(s)[0]


def test_simenv_step_horizon_and_velocity():
    s = _standing_state()
    nxt, steps, done = mo.simenv_step(s, np.zeros((1, 226), np.float32), np.array([298]))
    assert steps[0] == 299 and not done[0]
    nxt, steps, done = mo.simenv_step(s, np.zeros((1, 226), np.float32), np.array([299]))
    assert done[0]
    d = np.zeros((1, 226), np.float32)
    d[0, 200] = 101.0
    assert not mo.simenv_step(s, d, np.array([0]))[2][0]
    assert mo.simenv_step(s, d, np.array([0]), enable_velocity_check=True)[2][0]
    assert nxt.dtype == np.float64


# ---------------------------------------------------------------------------------------------------
# SimEnv against the reference's own sim_env.py (tests/golden/simenv_golden.npz, written by
# tests/golden/make_simenv_golden.py: the reference class run unmodified over stubbed gym / simulator imports)

def _simenv_golden():
    return np.load(os.path.join(os.path.dirname(__file__), "golden", "simenv_golden.npz"))


def test_simenv_tables_match_the_reference_constructor():
    """sim_env.py:84-116 with the reference's spinkick arg / character / controller files."""
    g = _simenv_golden()
    assert list(g["fall_offsets"]) == [9 * b + 1 for b in mo.HUMANOID3D_FALL_BODIES]
    for i, b in enumerate(mo.HUMANOID3D_FALL_BODIES):
        shape, p0, p1 = mo.HUMANOID3D_BODY_DEFS[b]
        assert (shape == "capsule") == bool(g["fall_is_capsule"][i])
        assert (p0, p1) == (g["fall_params"][i, 0], g["fall_params"][i, 1])
    assert int(g["record_all_world"]) == 0 and int(g["record_world_root_pos"]) == 0


def test_simenv_contact_thresholds_match_the_reference():
    """116 states placed 2e-6 / 1e-3 either side of `<= radius + 1e-4` for every fall body and both capsule caps."""
    g = _simenv_golden()
    got = mo.simenv_collided(g["contact_states"])
    assert (got == g["contact_collided"]).all()
    assert 0 < g["contact_collided"].sum() < g["contact_collided"].size


def test_simenv_velocity_check_matches_the_reference():
    g = _simenv_golden()
    zero = np.zeros_like(g["vel_states"], dtype=np.float32)
    steps = np.zeros(len(zero), dtype=np.int64)
    assert (mo.simenv_step(g["vel_states"], zero, steps, enable_velocity_check=True)[2] == g["vel_done_enabled"]).all()
    assert (mo.simenv_step(g["vel_states"], zero, steps)[2] == g["vel_done_default"]).all()
    assert g["vel_done_enabled"].any() and not g["vel_done_default"].any()


def test_simenv_controller_flags_match_the_reference():
    """RecordAllWorld / RecordWorldRootPos (sim_env.py:181-186, 224-231) and RecordVelAsPos (sim_env.py:264-267) set
    on the constructed reference object; 48 states per flag set with one fall body 2e-6 / 1e-3 off its threshold."""
    g = _simenv_golden()
    for k, (aw, wrp) in enumerate(g["variant_flag_sets"]):
        got = mo.simenv_collided(g["variant_states"][k], record_all_world=bool(aw), record_world_root_pos=bool(wrp))
        assert (got == g["variant_collided"][k]).all(), (aw, wrp)
        assert 0 < g["variant_collided"][k].sum() < 48
    got = mo.simenv_velocity_exploded(g["velpos_states"], divisor=float(g["velpos_divisor"]))
    assert (got == g["velpos_done"]).all() and g["velpos_done"].any() and not g["velpos_done"].all()


def test_simenv_episodes_match_the_reference():
    """reset -> 10 steps, five episodes, horizon 8: observations, step counter, done flags and the member
    round-robin of the reference SimEnv, replayed by the oracle (ensemble rebuilt from the seed and checked
    against the stored weight checksums)."""
    g = _simenv_golden()
    N, hidden = int(g["N"]), [int(h) for h in g["hidden"]]
    s, a, s2 = H.synth_dataset(int(g["dataset_rows"]), 226, 28, int(g["dataset_seed"]))
    ws, bs = mo.init_ensemble(226, 28, hidden, N, base_seed=int(g["base_seed"]), dense_connect=True)
    np.testing.assert_allclose([[float(w.double().abs().sum()) for w in m] for m in ws], g["weight_checksum"], rtol=1e-12)
    tf = mo.get_transformations(s, a, s2)
    assert list(g["traj_member"]) == [(e + 1) % N for e in range(len(g["traj_member"]))]   # sim_env.py:282-283
    for e in range(g["traj_ob0"].shape[0]):
        ob = g["traj_ob0"][e:e + 1].copy()
        m = int(g["traj_member"][e])
        steps = np.zeros(1, dtype=np.int64)
        for k in range(g["traj_actions"].shape[1]):
            act = torch.from_numpy(g["traj_actions"][e, k:k + 1]).float()
            preds = mo.ensemble_forward(ws, bs, tf, torch.from_numpy(ob).float(), act)
            ob, steps, done = mo.simenv_step(ob, preds[m].numpy(), steps, horizon=8)
            np.testing.assert_allclose(ob[0], g["traj_obs"][e, k], rtol=0, atol=1e-5)
            assert int(steps[0]) == int(g["traj_num_steps"][e, k]) and bool(done[0]) == bool(g["traj_done"][e, k])


# ---------------------------------------------------------------------------------------------------
# MLPCost (linear_cost.py:154-301) against the reference's own outputs (tests/golden/mlpcost_golden.npz)

MLPCOST_CASES = ["two_hidden", "one_hidden_quirk", "three_tanh"]


def _mlpcost_golden():
    import os
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "mlpcost_golden.npz"))


@pytest.mark.parametrize("tag", MLPCOST_CASES)
def test_mlp_cost_oracle_matches_reference(tag):
    g = _mlpcost_golden()
    expert = torch.from_numpy(g["expert"])
    oc = mo.MlpCostOracle(expert, hidden_dims=g[f"{tag}/hidden"].tolist(), activation=str(g[f"{tag}/act"]),
                          feature_dim=int(g[f"{tag}/feature_dim"]), input_type="ss", bw_quantile=0.1, lambda_b=0.3,
                          seed=100)
    assert len(oc.ws) == int(g[f"{tag}/n_linear"])
    for i, (w, b) in enumerate(zip(oc.ws, oc.bs)):  # same RNG stream -> the same net, bit for bit
        assert np.array_equal(w.numpy(), g[f"{tag}/w{i}"]) and np.array_equal(b.numpy(), g[f"{tag}/b{i}"])
    assert oc.bw == float(g[f"{tag}/bw"])
    xs, xa, nxt = (torch.from_numpy(g[k]) for k in ("xs", "xa", "next"))
    pi = torch.cat([xs, nxt], dim=1)
    assert np.array_equal(oc.phi_e.numpy(), g[f"{tag}/phi_e"])
    assert np.array_equal(oc.get_rep(pi).numpy(), g[f"{tag}/rep"])
    assert oc.fit_cost(pi) == float(g[f"{tag}/mmd"])
    assert np.array_equal(oc.get_costs(pi).numpy(), g[f"{tag}/costs"])
    assert float(oc.get_expert_cost()) == float(g[f"{tag}/expert_cost"])
    total, info = oc.get_bonus_costs(xs, xa, torch.from_numpy(g["disc"]), 0.4, next_states=nxt)
    assert np.array_equal(total.numpy(), g[f"{tag}/total"])
    for k in ("bonus", "ipm", "v_targ", "cost"):
        assert np.array_equal(info[k].numpy(), g[f"{tag}/info_{k}"]), k


# ---------------------------------------------------------------------------------------------------
# GAILCost evaluation side (gail_cost.py:18-43, 232-283) against the reference's own outputs

GAIL_CASES = ["ls_two_hidden", "ll_small", "ls_linear"]


def _gail_golden():
    import os
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "gail_golden.npz"))


@pytest.mark.parametrize("tag", GAIL_CASES)
def test_gail_cost_oracle_matches_reference(tag):
    g = _gail_golden()
    n = int(g[f"{tag}/n_linear"])
    ws = [torch.from_numpy(g[f"{tag}/w{i}"]) for i in range(n)]
    bs = [torch.from_numpy(g[f"{tag}/b{i}"]) for i in range(n)]
    ss = torch.cat([torch.from_numpy(g["xs"]), torch.from_numpy(g["next"])], dim=1)
    d = mo.gail_disc_forward(ws, bs, ss)
    assert np.array_equal(d.numpy(), g[f"{tag}/disc_outs"])
    c = mo.gail_costs(d.clone(), str(g[f"{tag}/loss_type"]))
    assert np.array_equal(c.numpy(), g[f"{tag}/costs"])
    total, info = mo.gail_bonus_costs(c, torch.from_numpy(g["disc"]), float(g[f"{tag}/lambda_b"]))
    assert np.array_equal(total.numpy(), g[f"{tag}/total"])
    for k in ("bonus", "ipm", "v_targ", "cost"):
        assert np.array_equal(info[k].numpy(), g[f"{tag}/info_{k}"]), k


# ---------------------------------------------------------------------------------------------------
# DynamicsModel.train_step (dynamics.py:236-250) against the reference's own three steps


def _train_golden():
    import os
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "train_golden.npz"))


def train_case(g, tag):
    dims = g[f"{tag}/dims"].tolist()
    S, A, N, dense, B = dims[:5]
    hidden = dims[5:]
    nl = len(hidden) + 1
    tf = tuple(torch.from_numpy(g[f"{tag}/tf{i}"]) for i in range(6))
    optim = {"optim": str(g[f"{tag}/optim"]), "lr": float(g[f"{tag}/lr"]), "momentum": 0.9, "eps": 1e-8}
    ws = [[torch.from_numpy(g[f"{tag}/init/m{k}/fc_layers.{l}.weight"]) for l in range(nl)] for k in range(N)]
    bs = [[torch.from_numpy(g[f"{tag}/init/m{k}/fc_layers.{l}.bias"]) for l in range(nl)] for k in range(N)]
    data = tuple(torch.from_numpy(g[k]) for k in ("ds_s", "ds_a", "ds_s2"))
    return dict(S=S, A=A, N=N, dense=bool(dense), B=B, hidden=hidden, nl=nl, tf=tf, optim=optim, ws=ws, bs=bs,
                act=str(g[f"{tag}/act"]), clip=float(g[f"{tag}/clip"]), idx=torch.from_numpy(g["idx"]), data=data)


@pytest.mark.parametrize("tag", ["sgd_dense", "adam_plain_tanh"])
def test_train_oracle_matches_reference(tag):
    g = _train_golden()
    c = train_case(g, tag)
    s, a, s2 = c["data"]
    for k in range(c["N"]):
        o = mo.TrainOracle(c["ws"][k], c["bs"][k], c["tf"], c["dense"], c["act"], c["optim"])
        bi = c["idx"][0, k]
        assert o.validate_step(s[bi], a[bi], s2[bi]) == float(g[f"{tag}/val0/m{k}"])
        o.grads(s[bi], a[bi], s2[bi])
        for l in range(c["nl"]):
            assert np.array_equal(o.ws[l].grad.numpy(), g[f"{tag}/grad0/m{k}/fc_layers.{l}.weight"])
            assert np.array_equal(o.bs[l].grad.numpy(), g[f"{tag}/grad0/m{k}/fc_layers.{l}.bias"])
        for step in range(3):
            bi = c["idx"][step, k]
            loss = o.train_step(c["clip"], s[bi], a[bi], s2[bi])
            assert loss == float(g[f"{tag}/loss/m{k}"][step])
            for l in range(c["nl"]):
                assert np.array_equal(o.ws[l].detach().numpy(), g[f"{tag}/step{step}/m{k}/fc_layers.{l}.weight"])
                assert np.array_equal(o.bs[l].detach().numpy(), g[f"{tag}/step{step}/m{k}/fc_layers.{l}.bias"])
