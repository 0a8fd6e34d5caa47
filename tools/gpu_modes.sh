#!/bin/bash
# the documented run-time knobs still pass the parity suite's core: f16x3 (three fp16 passes), simt (fp32 FFMA twin), no graphs / no PDL
mkdir -p gpurun_out
CORE="small_model or edge or odd_dim or config2 or forward or sample_rl_logprobs or indexed"
for cfg in "f16x3:VSRDEC_GEMM=f16x3" "simt:VSRDEC_GEMM=simt" "nograph:VSRDEC_GRAPH=0 VSRDEC_PDL=0"; do
  name=${cfg%%:*}; envs=${cfg#*:}
  SEL="$CORE"; [ $name = simt ] && SEL="($CORE) and not half_features"    # the FFMA twin takes fp32 features only
  env $envs timeout 900 python -m pytest tests -m gpu -q -x -k "$SEL" > gpurun_out/modes_$name.log 2>&1
  echo "$name rc=$?: $(tail -1 gpurun_out/modes_$name.log)"
done
