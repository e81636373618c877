#!/bin/bash
# experiment: lanes per env of env_kernel (CM_ENV_GROUP; 0 = the library's own choice) at the team sizes of C3 / C4 / C5
# usage: gpurun -- 'bash tools/env_group_sweep.sh'      (library builds are compared with tools/variant_sweep.sh)
# measures speed only; bit-exactness under every group is tests/test_gpu_env_layouts.py (each group forced in its own process)
mkdir -p gpurun_out
run() {  # config group
  CM_ENV_GROUP=$2 python bench.py --config $1 --no-cpu-baseline --no-sweep --e2e-steps 4 2>/dev/null | python -c "
import json,sys
d=json.loads(sys.stdin.read().strip().splitlines()[-1])
print('$1 group $2', 'value %.1fM' % (d['value']/1e6), 'ms/step %.4f' % d['ms_per_step'], 'policy %.4f' % d['roofline']['ms_per_launch'], 'env %.4f (alone %.4f)' % (d['roofline_env']['ms_per_launch'], d['roofline_env'].get('ms_per_launch_alone', 0)))"
}
{
for spec in "c3 0" "c3 4" "c3 8" "c3 16" "c3 32" "c4 0" "c4 16" "c4 32" "c5 0" "c5 16" "c1 0" "c2 0"; do run $spec; done
python -m pytest tests/test_gpu_env.py tests/test_gpu_fullsize.py tests/test_gpu_rollout.py -m gpu -x -q 2>&1 | tail -3
} | tee gpurun_out/env_group_sweep.txt
