"""Writes the outputs of the env step + cost for a set of batch sizes to an .npz (python write_step_outputs.py OUT).
tests/test_parity_gpu.py runs it once with SIMSTEP_CHAIN=0 (one launch per layer) and once with the column-fused
forward kernel, in two processes because the switch is read once per process, and compares the two files."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main(out_path):
    from oracle import milo_oracle as mo
    from tests import helpers as H
    from amp_extensions_b200.engine import Engine, HumanoidTermination
    c = H.ns_case()
    eng = Engine(c["S"], c["A"], c["N"], c["hidden"], dense_connect=True, activation="relu", transform=True,
                 precision="fp16")
    eng.load_ensemble(c["ws"], c["bs"], c["tf"])
    eng.set_termination(HumanoidTermination(enable_velocity_check=True))
    oc = mo.RffCostOracle(H.ns_expert(), feature_dim=512, input_type="ss", bw_quantile=0.1, lambda_b=0.0025, seed=100)
    g = torch.Generator().manual_seed(5)
    oc.w = torch.randn(512, generator=g) * 0.01
    eng.load_rff(oc.rff_weight, oc.rff_bias, split=True)
    res = {}
    # 4 800 and 40 001 rows end in a shared last round of the column-fused kernel, 7 000 and 21 500 in a plain one
    for E in (1, 127, 2000, 4800, 7000, 21500, 40001):
        s = H.humanoid_like_states(E, seed=70 + E % 7)
        a = torch.randn(E, 28, generator=g)
        member = torch.randint(0, 4, (E,), generator=g, dtype=torch.int32)
        if E > 100:
            member[3] = 7          # out of range: the row's next state must be NaN on both paths
        steps = torch.randint(0, 300, (E,), generator=g, dtype=torch.int32).cuda()
        for split in (True, False):
            eng.set_rff_split(split)
            st = steps.clone()
            out = eng.step_cost(s.cuda(), a.cuda(), member.cuda(), st, oc.w.cuda(), 0.0025, c["threshold"])
            for name, t in zip(("next", "disc", "done", "cost", "ipm", "bonus"), out):
                res[f"E{E}_s{int(split)}_{name}"] = t.cpu().numpy()
            res[f"E{E}_s{int(split)}_steps"] = st.cpu().numpy()
        d = eng.discrepancy(s, a)
        res[f"E{E}_disc_only"] = d.cpu().numpy()
    # a second, irregular ensemble: three members, NO dense connections, tanh, hidden sizes 512 / 256 / 512 (2, 1 and 2
    # n-tiles: the two pairs that share a unit of the last round get unequal work), batch sizes that give the column-fused
    # kernel shared units without (6 812 rows) and with (19 193 rows) whole rounds of members in sequence
    from oracle import milo_oracle as mo2
    S2, A2, N2, hid2 = 226, 28, 3, [512, 256, 512]
    ws2, bs2 = mo2.init_ensemble(S2, A2, hid2, N2, dense_connect=False, base_seed=7)
    eng2 = Engine(S2, A2, N2, hid2, dense_connect=False, activation="tanh", transform=True, precision="fp16")
    eng2.load_ensemble(ws2, bs2, c["tf"])
    eng2.set_termination(HumanoidTermination(enable_velocity_check=False))
    for E in (6812, 19193):
        s = H.humanoid_like_states(E, seed=E % 11)
        a = torch.randn(E, 28, generator=g)
        member = torch.randint(0, N2, (E,), generator=g, dtype=torch.int32)
        st = torch.zeros(E, dtype=torch.int32).cuda()
        out = eng2.step(s.cuda(), a.cuda(), member.cuda(), st)
        for name, t in zip(("next", "disc", "done"), out):
            res[f"plain_E{E}_{name}"] = t.cpu().numpy()
        res[f"plain_E{E}_steps"] = st.cpu().numpy()
    np.savez(out_path, **res)


if __name__ == "__main__":
    main(sys.argv[1])
