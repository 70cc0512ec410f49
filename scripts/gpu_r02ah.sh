#!/bin/bash
set -u
mkdir -p gpurun_out
TAG=${1:-r02ah}
echo "== pytest -m gpu"; timeout 1200 python -m pytest tests -q -m gpu -x > gpurun_out/${TAG}_pytest.log 2>&1; echo "pytest exit $?"; tail -4 gpurun_out/${TAG}_pytest.log
echo "== bench"; timeout 900 python bench.py --no-ref-ext --no-cpu-baseline > gpurun_out/${TAG}_bench.json 2>gpurun_out/${TAG}_bench.err; python -c "
import json; d=json.load(open('gpurun_out/${TAG}_bench.json')); print(d['value'], d['ms_per_step'], d['loop']['ms_per_iteration'], d['loop']['pose_only']['ms_per_iteration'], d['e2e']['ms_per_step'], d['roofline']['launch_ms'])"
