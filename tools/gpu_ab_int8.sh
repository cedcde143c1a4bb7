#!/bin/bash
# Same-box A/B runs of the INT8 route's knobs (run on the GPU box from the repo root, one gpurun call; DESIGN.md section 8 quotes
# their results).  Each line is one short bench (10 steps after 3 warm-up steps, no extras) or one pass of the grid prediction.
llh() { python bench.py --steps 10 --warmup 3 --no-extra --no-cpu --grid-points 3e5 2>/dev/null | python -c "
import json,sys
d=json.loads(sys.stdin.read().strip().splitlines()[-1]); r=d['roofline']['by_kernel_ms_per_step']
print('evals/s',round(d['value'],1),'ms/step',round(d['ms_per_step'],2),{k:round(v,2) for k,v in r.items() if v})"; }
pred() { timeout 300 python tools/perf_pred.py 2000 8 4194304 2>&1 | tail -n 1; }
echo "--- default";                       llh; pred
echo "--- FP64 DMMA everywhere";          GPE_OZAKI=0 llh; GPE_OZAKI=0 pred
echo "--- 14 moduli";                     GPE_OZAKI=14 llh; GPE_OZAKI=14 pred
echo "--- INT8 from 512 up";              GPE_OZAKI_MIN=512 llh
echo "--- one / four sub-batch groups";   GPE_OZAKI_STREAMS=1 llh; GPE_OZAKI_STREAMS=4 llh
echo "--- default";                       llh; pred
