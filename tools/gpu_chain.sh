#!/bin/bash
# column-fused forward (gemm_chain.cuh) against one launch per layer: bitwise comparison of the step's outputs, then a
# short bench of each (SIMSTEP_CHAIN=0: one launch per layer; 2: the default).  Usage: bash tools/gpu_chain.sh [tag]
TAG=${1:-chain}
OUT=gpurun_out; mkdir -p $OUT
for m in 0 2; do
  SIMSTEP_CHAIN=$m timeout 300 python tests/write_step_outputs.py /tmp/c$m.npz 2>&1 | tail -5 || echo "mode $m run failed"
done
python - <<'PY'
import numpy as np
a, b = np.load("/tmp/c0.npz"), np.load("/tmp/c2.npz")
bad = [k for k in a.files if not np.array_equal(a[k], b[k], equal_nan=True)]
print("bitwise identical" if not bad else "DIFFERS in %s" % bad[:8])
for k in bad[:4]:
    print("  ", k, float(np.nanmax(np.abs(a[k].astype(np.float64) - b[k].astype(np.float64)))))
PY
for m in 0 2; do
for i in 1 2; do
SIMSTEP_CHAIN=$m timeout 300 python bench.py --steps 50 --warmup 5 --skip-cpu-baseline --skip-e2e --skip-sustained --skip-extras > $OUT/${TAG}_m${m}_$i.json 2> $OUT/${TAG}_m${m}_$i.err
python - <<PY
import json
try:
    d = json.loads(open("$OUT/${TAG}_m${m}_$i.json").read().strip().splitlines()[-1])
    print("mode $m run $i", "value %.4g ms %.4f" % (d["value"], d["ms_per_step"]), {k: round(v, 4) for k, v in d.get("kernels_ms_per_step").items()})
except Exception as e:
    print("mode $m failed", e); print(open("$OUT/${TAG}_m${m}_$i.err").read()[-1500:])
PY
done
done
