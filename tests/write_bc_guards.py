"""Runs one DeviceBC fit (MLE, two epochs, batch 65 with a ragged last tile) at every policy shape of tests/test_bc_gpu.py
and writes each handle's guard-zone check, before the BC state exists and after the fit, to an .npz
(python write_bc_guards.py OUT).  The test runs it under SIMSTEP_DEBUG_GUARDS=1 in a process of its own because the
library reads that switch when a handle is created."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main(out_path):
    import torch
    from amp_extensions_b200.bc import DeviceBC
    from tests import test_policy_matrix_gpu as M
    from tests import test_bc_gpu as T
    res = {}
    for cid in T.IDS:
        cd = M.case_data(cid)
        eng = M.engine()
        M.load(eng, cd)
        n0, _ = eng.check_guards()
        bc = DeviceBC(eng, M.host_policy(cd, cd["theta"]), epochs=2, batch_size=65, loss_type="MLE")
        obs, act = cd["obs"][:1000].cuda(), cd["act"][:1000].cuda()
        bc.fit_tensors(obs, act, return_losses=True)
        torch.cuda.synchronize()
        n1, bad = eng.check_guards()
        res[cid] = np.array([n0, n1, bad])
        eng.close()
    np.savez(out_path, **res)


if __name__ == "__main__":
    main(sys.argv[1])
