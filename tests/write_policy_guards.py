"""Runs one DeviceNPG update (valid mask, HVP subsample) at every case of tests/test_policy_matrix_gpu.py's table and
writes each handle's guard-zone check, before the NPG state exists and after the update, to an .npz
(python write_policy_guards.py OUT).  The test runs it under SIMSTEP_DEBUG_GUARDS=1 in a process of its own because the
library reads that switch when a handle is created."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main(out_path):
    import torch
    from amp_extensions_b200.npg import DeviceNPG
    from tests import test_policy_matrix_gpu as M
    res = {}
    for c in M.CASES:
        cd = M.case_data(c["id"])
        n = M.row_counts(cd["q"]["R"])[-1]
        eng = M.engine()
        M.load(eng, cd)
        n0, _ = eng.check_guards()
        npg = DeviceNPG(eng, M.host_policy(cd, cd["theta"]), hvp_sample_frac=0.5)
        valid = (torch.arange(n) % 3 != 0).to(torch.uint8).cuda()
        npg.update((cd["obs"][:n].cuda(), cd["act"][:n].cuda()), cd["adv"][:n].cuda(), valid)
        n1, bad = eng.check_guards()
        res[c["id"]] = np.array([n0, n1, bad])
        eng.close()
    np.savez(out_path, **res)


if __name__ == "__main__":
    main(sys.argv[1])
