#!/bin/bash
# Alternating A/B of libecb.so builds in one process tree on one GPU: the variants take turns, <rounds> times each, so that
# clock and neighbour drift hit all of them alike.  One JSON line per run: step time, k_cluster's CUDA-event time, e2e, clocks.
#   profiles/tools/ab_alternate.sh <out.jsonl> <rounds> <config> <tag>=<libecb.so> [<tag>=<libecb.so> ...]
# (a parent build for <tag>: git worktree add /tmp/parent <commit> && python -m eventcalib_b200.build there)
out=$1; rounds=$2; config=$3; shift 3
: > "$out"
gpu=$(nvidia-smi --query-gpu=name,power.limit --format=csv,noheader | head -1)
for r in $(seq "$rounds"); do
  for v in "$@"; do
    tag=${v%%=*}; lib=$(realpath "${v#*=}")
    ECB_LIBRARY=$lib python bench.py --gpus 1 --config "$config" --no-cpu --steps 20 --warmup 5 2>/dev/null | \
      TAG=$tag ROUND=$r CONFIG=$config GPU="$gpu" python -c "
import json, os, sys
d = json.loads(sys.stdin.read().strip().splitlines()[-1])
k = d['roofline']['kernels']
print(json.dumps({'variant': os.environ['TAG'], 'round': int(os.environ['ROUND']), 'config': os.environ['CONFIG'],
                  'gpu': os.environ['GPU'], 'ms_per_step': d['ms_per_step'], 'cluster_ms': k['cluster']['ms'],
                  'e2e_ms': d['e2e']['ms_per_step'], 'clocks': d['clocks'],
                  'stages': {s: round(v['ms'], 4) for s, v in k.items()}}))" | tee -a "$out"
  done
done
