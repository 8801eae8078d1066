"""Writes the step and step-cost outputs of every case of tests/test_step_matrix_gpu.py's table to an .npz (python
write_matrix_outputs.py OUT), with each handle's forward launch count and guard-zone check.  The tests run it with and
without SIMSTEP_CHAIN=0 and under SIMSTEP_DEBUG_GUARDS=1, in processes of their own because the library reads both
switches once per process."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main(out_path):
    from tests import test_step_matrix_gpu as M
    res = {}
    for c in M.CASES:
        cd = M.case_data(c["id"])
        oc, _ = M.cost_oracle(cd, "ss", 100)
        for prec in ("tf32", "fp16"):
            eng = M.engine(c["id"], prec)
            eng.load_rff(oc.rff_weight, oc.rff_bias, split=True, input_type="ss")
            tag = f"{c['id']}_{prec}"
            launches = []
            for E in (257, 1029):
                s, a, member, steps = M.inputs(cd, E, seed=9)
                sd, ad, md = s.cuda(), a.cuda(), member.cuda()
                st = steps.clone().cuda()
                for name, t in zip(("next", "disc", "done"), eng.step(sd, ad, md, st)):
                    res[f"{tag}_E{E}_step_{name}"] = t.cpu().numpy()
                res[f"{tag}_E{E}_step_steps"] = st.cpu().numpy()
                for split in (True, False):
                    eng.set_rff_split(split)
                    out = eng.step_cost(sd, ad, md, steps.clone().cuda(), oc.w.cuda(), 0.3, 0.5)
                    for name, t in zip(("next", "disc", "done", "cost", "ipm", "bonus"), out):
                        res[f"{tag}_E{E}_cost{int(split)}_{name}"] = t.cpu().numpy()
                launches.append(eng.forward_launches(E))
            res[f"launches_{tag}"] = np.array(launches)
            res[f"guards_{tag}"] = np.array(eng.check_guards())
            eng.close()
    np.savez(out_path, **res)


if __name__ == "__main__":
    main(sys.argv[1])
