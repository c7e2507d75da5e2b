#!/bin/bash
# Round 5a, GPU call 2: the path-query tests again, after call 1 called for two fixes in the oracle comparison (a point light's
# intensity is compared to the record bar, not bit for bit; an empty set of light entries passes).
#   tools/gpu_calls/r5a_call02.sh OUTPUT_DIR
out=${1:?usage: r5a_call02.sh OUTPUT_DIR}
cd "$(dirname "$0")/../.."
mkdir -p "$out"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader > "$out"/card.txt 2>&1
timeout 300 python -c "import __graft_entry__ as g; g.build(verbose=False)" > "$out"/build.log 2>&1; echo "build rc=$?" >> "$out"/build.log
timeout 1500 python -m pytest -q -m gpu -rs -s tests/test_gpu_path_queries.py > "$out"/gpu_paths.log 2>&1; echo "gpu_paths rc=$?" >> "$out"/gpu_paths.log
tail -n 3 "$out"/build.log "$out"/gpu_paths.log
