#!/bin/bash
# round 3: the fused expand + depthwise kernel (expdw_kernel) in one command - build, GPU tests, alternating A/B bench runs
# (default vs MTB_EXPDW=0, the two-launch path), op profiles of both, one full default bench line.
# Usage: scripts/r3/gpu_expdw.sh <output dir>
OUT=${1:?usage: $0 <output dir>}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/smi.txt" 2>&1
python -c "import __graft_entry__ as g; g.build()" > "$OUT/build.log" 2>&1 || { echo "build failed"; tail -20 "$OUT/build.log"; exit 1; }
timeout 900 python -m pytest tests/test_gpu_expdw.py tests/test_host_expdw.py -q -s -x > "$OUT/tests_expdw.log" 2>&1
rc=$?
echo "expdw tests exit $rc" >> "$OUT/tests_expdw.log"
tail -15 "$OUT/tests_expdw.log"
[ $rc -eq 0 ] || exit 1
python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/smoke.log" 2>&1; echo "smoke exit $?" >> "$OUT/smoke.log"
timeout 1500 python -m pytest tests -m gpu -q > "$OUT/tests_gpu.log" 2>&1; echo "gpu suite exit $?" >> "$OUT/tests_gpu.log"
timeout 600 python -m pytest tests -q -m "not gpu" > "$OUT/tests_cpu.log" 2>&1; echo "cpu suite exit $?" >> "$OUT/tests_cpu.log"
for i in 1 2 3; do
  for arm in fused unfused; do
    if [ $arm = unfused ]; then export MTB_EXPDW=0; else unset MTB_EXPDW; fi
    timeout 600 python bench.py --steps 50 --no-cpu-baseline --no-frames --no-parity-line --dump-outputs "$OUT/dump_${arm}_$i" \
      > "$OUT/bench_${arm}_$i.json" 2> "$OUT/bench_${arm}_$i.err"
  done
done
unset MTB_EXPDW
timeout 600 python scripts/op_profile.py --batch 256 > "$OUT/op_profile_fused_b256.txt" 2>&1
MTB_EXPDW=0 timeout 600 python scripts/op_profile.py --batch 256 > "$OUT/op_profile_unfused_b256.txt" 2>&1
timeout 1200 python bench.py > "$OUT/bench_full.json" 2> "$OUT/bench_full.err"
python - "$OUT" <<'PY'
import glob, json, os, sys
import numpy as np
out = sys.argv[1]
ms = {}
for arm in ('fused', 'unfused'):
    for f in sorted(glob.glob(f'{out}/bench_{arm}_*.json')):
        for line in open(f):
            if line.startswith('{'):
                ms.setdefault(arm, []).append(json.loads(line).get('ms_per_step'))
print('ms_per_step', ms)
d = sorted(glob.glob(f'{out}/dump_*/coords3d_abs.npy'))
a = [np.load(x) for x in d]
print('dumps', len(a), 'all identical:', all(np.array_equal(a[0], x) for x in a[1:]))
PY
tail -n 3 "$OUT/tests_gpu.log" "$OUT/smoke.log" "$OUT/tests_cpu.log"
