#!/bin/bash
# Quick K2 check on the GPU box: the tests that exercise the coded E-step, then one short bench line.
#   bash scripts/k2_quick.sh
python -m pytest tests -m gpu -q -x -k "${K2_TESTS:-code_pass}" 2>&1 | tail -3
python bench.py --steps 20 --warmup 3 --no-cpu-baseline --no-cfg4 --no-k1 --replicas 0 2>/dev/null | python -c "
import json,sys
d=json.load(sys.stdin)
k=d['kernels']['K2_estep_qF_coded']
print('K2 mean %.4f (min %.4f med %.4f max %.4f) ms frac %.3f  ms/step %.3f steady %.3f share %.2f'%(k['mean_ms'],k.get('min_ms',0),k.get('median_ms',0),k.get('max_ms',0),k['frac_of_hbm_peak'],d['ms_per_step'],d['steady_state']['ms_per_step'],d['kernel_share_of_step']))
for k,v in d['kernels'].items(): print('%-22s %4d  %.4f ms (min %.4f med %.4f max %.4f) share %.3f'%(k, v['launches'], v['mean_ms'], v.get('min_ms',0), v.get('median_ms',0), v.get('max_ms',0), v['share_of_step']))
"
