#!/usr/bin/env bash
# Quick check of a kernel change: parity suite, then kernel timings of this build.
#   bash tools/gpu_quick.sh <tag> ["<pytest -k expression>"]
set -u
TAG="${1:-q}"; KEXPR="${2:-}"
O=gpurun_out/$TAG; mkdir -p "$O"
if [ -n "$KEXPR" ]; then timeout 1200 python -m pytest tests -m gpu -q -k "$KEXPR" > "$O/pytest_gpu.log" 2>&1
else timeout 1200 python -m pytest tests -m gpu -q > "$O/pytest_gpu.log" 2>&1; fi
echo "pytest rc=$?" >> "$O/pytest_gpu.log"
grep -E "^(FAILED|ERROR)|passed|failed|rc=" "$O/pytest_gpu.log" | tail -25
for cfg in "--config C2 --sites 1000000" "--config C3 --sites 100000" "--config C5 --sites 1000000" "--config C4 --sites 9472"; do
  echo "$cfg" | tee -a "$O/run_kernel.log"
  timeout 300 python tools/run_kernel.py $cfg --launches 5 2>&1 | tee -a "$O/run_kernel.log"
done
