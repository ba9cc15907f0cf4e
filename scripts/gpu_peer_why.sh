#!/bin/bash
# where does the peer-halo overhead on THICK fp64 slabs come from?  (2 GPUs)
mkdir -p gpurun_out
TR="python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1"
python scripts/peer_codegen_check.py c4 > gpurun_out/r2_peer_codegen_c4_idle.json 2> gpurun_out/r2_peer_codegen_c4_idle.err; cat gpurun_out/r2_peer_codegen_c4_idle.json
run() {  # tag, env, args
  timeout 420 env $2 $TR --master-port 2954$((RANDOM % 10)) scripts/check_peer_halo.py $3 > gpurun_out/r2_peerwhy_$1.log 2>&1
  echo "== $1 ($2 $3) rc=$?"; grep "^{\|Error" gpurun_out/r2_peerwhy_$1.log | tail -3
}
run c4_768_memset "PSAD_CHECK_SHAPE=768,768,768 PSAD_PEER_STREAM_SIGNAL=1" "c4 zeros 3 --time"
