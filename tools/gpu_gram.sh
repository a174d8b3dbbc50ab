#!/bin/bash
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
TAG=${1:-x}
timeout 900 python -m pytest tests/test_gpu_parity.py -x -q -m gpu -k "gram or ahead or bench_geometry or float64_loader or variant" 2>&1 | tail -3
timeout 300 python bench.py --steps 20 --warmup 3 --no-e2e --no-cpu 2>gpurun_out/gram_${TAG}.err | python -c "
import json,sys
d=json.loads(sys.stdin.read().strip().splitlines()[-1]); print('bench ->', round(d['ms_per_step'],4), {k: round(v,4) for k,v in d['roofline']['kernel_ms'].items()})"
