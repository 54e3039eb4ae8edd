#!/bin/bash
# A/B of k_fused builds on one box: scripts/kb_mel.py for every variant given as
# name=path[,ENV=VALUE...] (default build when path is empty), interleaved three times.
# usage: scripts/ab_mel.sh old=challenge_b200/build_old/libiris.so generic=,IRIS_NO_FIXED_EPI=1 new=
mkdir -p gpurun_out
: > gpurun_out/ab_mel.log
for rep in 1 2 3; do
  for spec in "$@"; do
    name=${spec%%=*}; rest=${spec#*=}
    path=${rest%%,*}; envs=""
    if [[ "$rest" == *,* ]]; then envs=${rest#*,}; fi
    (
      if [ -n "$path" ]; then export IRIS_LIB=$PWD/$path; fi
      IFS=',' read -ra kv <<< "$envs"
      for e in "${kv[@]}"; do [ -n "$e" ] && export "$e"; done
      echo -n "$name: " >> gpurun_out/ab_mel.log
      timeout 300 python scripts/kb_mel.py 2>&1 | tail -1 >> gpurun_out/ab_mel.log
    )
  done
done
cat gpurun_out/ab_mel.log
