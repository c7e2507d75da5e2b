#!/bin/bash
# Round 4a, GPU call 2: the crossing tests again, after the fixes call 1 called for (the mesh walk's pop, two test bars).
#   tools/gpu_calls/r4a_call02.sh OUTPUT_DIR
out=${1:?usage: r4a_call02.sh OUTPUT_DIR}
cd "$(dirname "$0")/../.."
mkdir -p "$out"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader > "$out"/card.txt 2>&1
timeout 300 python -c "import __graft_entry__ as g; g.build(verbose=False)" > "$out"/build.log 2>&1; echo "build rc=$?" >> "$out"/build.log
timeout 1200 python -m pytest -q -m gpu -rs -s tests/test_gpu_ray_crossings.py > "$out"/gpu_crossings.log 2>&1
tail -n 3 "$out"/build.log "$out"/gpu_crossings.log
