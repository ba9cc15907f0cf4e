#!/bin/bash
# A/B at N ranks: what makes the per-kernel time at N > 1 differ from round 1 (1.42 ms at N=8)?  Each arm: headline only, no e2e.
N=${1:-4}
mkdir -p gpurun_out
R="python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1"
B="bench.py --gpus $N --steps 20 --warmup 5 --no-e2e"
i=0
for arm in "" "PSAD_BENCH_NO_NVML=1" "PSAD_NO_LAUNCH_CACHE=1" "" "PSAD_BENCH_NO_NVML=1"; do
  i=$((i+1))
  env $arm $R --master-port $((29530+i)) $B > gpurun_out/r2_ab_n${N}_$i.json 2> gpurun_out/r2_ab_n${N}_$i.err
  python - "$arm" gpurun_out/r2_ab_n${N}_$i.json <<'PY'
import json, sys
d = json.loads(open(sys.argv[2]).read().strip().splitlines()[-1])
r = d['roofline']
print('%-28s ms/step %.4f  fwd %.4f adj %.4f  host_issue %.3f  clocks %s' % (sys.argv[1] or '(shipped)', d['ms_per_step'], r['forward_ms'], r['adjoint_ms'], d['host_issue_ms_per_step'], d['clocks'].get('sm_min_mhz')))
PY
done
