#!/bin/bash
# Round 6a, GPU call 2: the final tree.  The card, a clean build of the CUDA library, the whole GPU suite, smoke() and bench.py.
# Everything is written under OUTPUT_DIR.
#   tools/gpu_calls/r6a_call02.sh OUTPUT_DIR
out=${1:?usage: r6a_call02.sh OUTPUT_DIR}
cd "$(dirname "$0")/../.."
mkdir -p "$out"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader > "$out"/card.txt 2>&1
make -C functracer_b200/csrc clean > /dev/null 2>&1
timeout 900 python -c "import __graft_entry__ as g; g.build(verbose=False)" > "$out"/build.log 2>&1; echo "build rc=$?" >> "$out"/build.log
timeout 2700 python -m pytest -q -m gpu -rs tests > "$out"/gpu_suite.log 2>&1; echo "gpu_suite rc=$?" >> "$out"/gpu_suite.log
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > "$out"/smoke.log 2>&1; echo "smoke rc=$?" >> "$out"/smoke.log
timeout 600 python bench.py --gpus 1 --steps 5 --warmup 2 > "$out"/bench_tree.json 2> "$out"/bench_tree.err
tail -n 3 "$out"/build.log "$out"/gpu_suite.log "$out"/smoke.log
head -c 400 "$out"/bench_tree.json
