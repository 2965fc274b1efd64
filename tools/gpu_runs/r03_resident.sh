#!/bin/bash
# resident-chain MLP kernel (csrc/gemm_resident.cuh): full GPU suite, smoke, and the bench with ANI_B200_MLP_RESIDENT=0
# (the data-flow launch / chained launches of the parent) against the default selection (arm "d"; =1 forces the resident
# kernel), water10k alternated three times, the other configs once per arm; the dumped outputs of the two arms compared.
# Usage: bash tools/gpu_runs/r03_resident.sh OUTPUT_DIR
O=${1:?usage: $0 OUTPUT_DIR}
mkdir -p $O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/r03_gpu.txt 2>&1; cat $O/r03_gpu.txt
timeout 120 python -m pytest tests/test_mlp_resident_plan.py -q -s > $O/r03_plan.log 2>&1; grep "resident plan" $O/r03_plan.log
timeout 1200 python -m pytest tests -m gpu -q > $O/r03_pytest.log 2>&1; echo "pytest rc=$?"; tail -4 $O/r03_pytest.log
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $O/r03_smoke.log 2>&1; echo "smoke rc=$?"; tail -1 $O/r03_smoke.log
bench() {   # config arm tag steps
  if [ "$2" = d ]; then unset ANI_B200_MLP_RESIDENT; else export ANI_B200_MLP_RESIDENT=$2; fi
  timeout 300 python bench.py --gpus 1 --steps $4 --warmup 20 --cpu-steps 0 --config $1 \
    --dump-outputs $O/r03_dump_$1_resident$2 > $O/r03_bench_$1_resident$2$3.json 2> $O/r03_bench_$1_resident$2$3.err
  echo -n "$1 resident=$2$3 rc=$? "; python -c "
import json; d=json.loads(open('$O/r03_bench_$1_resident$2$3.json').read().strip().splitlines()[-1])
print('ms_per_step %.4f mlp %.4f' % (d['ms_per_step'], d['stage_ms']['mlp_forward_backward']))"
}
for i in 1 2 3; do for arm in 0 d; do bench water10k $arm _$i 200; done; done
for cfg in water1k gdb256 protein50k; do for arm in 0 d; do bench $cfg $arm "" 100; done; done
python - "$O" <<'PY' 2>&1 | tee $O/r03_dump_compare.txt
import glob, os, sys
import numpy as np
out = sys.argv[1]
for cfg in ("water10k", "water1k", "gdb256", "protein50k"):
    a, b = f"{out}/r03_dump_{cfg}_resident0", f"{out}/r03_dump_{cfg}_residentd"
    for f in sorted(glob.glob(a + "/*.npy")):
        x, y = np.load(f).astype(np.float64), np.load(os.path.join(b, os.path.basename(f))).astype(np.float64)
        print(f"{cfg} {os.path.basename(f)} max|d| = {np.abs(x - y).max():.3e} (max |x| {np.abs(x).max():.3e})")
PY
unset ANI_B200_MLP_RESIDENT
rm -rf $O/r03_dump_*_resident?
