"""Runs train_grads and train_step at every case and batch size of tests/test_train_matrix_gpu.py's table and writes
each training handle's guard-zone check to an .npz (python write_train_guards.py OUT).  The test runs it under
SIMSTEP_DEBUG_GUARDS=1 in a process of its own because the library reads that switch when a handle is created."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main(out_path):
    from tests import test_train_matrix_gpu as M
    res = {}
    for c in M.CASES:
        cd = M.case_data(c["id"])
        for handle, cap, batches in (("max", M.MAX_ROWS, M.BATCH_ORDER), ("exact", M.EXACT, [M.EXACT])):
            eng = M.train_engine(cd, cap)
            for B in batches:
                s, a, s2 = M.cuda(*M.batch(cd, B))
                eng.train_grads(s, a, s2)
                eng.train_step(s, a, s2, grad_clip=1.0)
            res[f"{c['id']}_{handle}"] = np.array(eng.check_guards())
            eng.close()
    np.savez(out_path, **res)


if __name__ == "__main__":
    main(sys.argv[1])
