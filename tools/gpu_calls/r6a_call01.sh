#!/bin/bash
# Round 6a, GPU call 1: sample shading (ftb_frame_rays, ftb_shade_samples).  The card, the build, the new GPU tests, smoke(),
# bench.py, tools/sample_rate.py and the GPU tests of windows, lit tiles and path queries.  Everything is written under OUTPUT_DIR.
#   tools/gpu_calls/r6a_call01.sh OUTPUT_DIR
out=${1:?usage: r6a_call01.sh OUTPUT_DIR}
cd "$(dirname "$0")/../.."
mkdir -p "$out"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader > "$out"/card.txt 2>&1
timeout 300 python -c "import __graft_entry__ as g; g.build(verbose=False)" > "$out"/build.log 2>&1; echo "build rc=$?" >> "$out"/build.log
timeout 1500 python -m pytest -q -m gpu -rs -s tests/test_gpu_sample_shading.py > "$out"/gpu_samples.log 2>&1; echo "gpu_samples rc=$?" >> "$out"/gpu_samples.log
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > "$out"/smoke.log 2>&1; echo "smoke rc=$?" >> "$out"/smoke.log
timeout 600 python bench.py --gpus 1 --steps 5 --warmup 2 > "$out"/bench_tree.json 2> "$out"/bench_tree.err
timeout 900 python tools/sample_rate.py > "$out"/sample_rate.txt 2>&1; echo "sample_rate rc=$?" >> "$out"/sample_rate.txt
timeout 900 python -m pytest -q -m gpu tests/test_gpu_window.py tests/test_gpu_lit_tiles.py tests/test_gpu_path_queries.py > "$out"/gpu_some.log 2>&1; echo "gpu_some rc=$?" >> "$out"/gpu_some.log
tail -n 3 "$out"/build.log "$out"/gpu_samples.log "$out"/smoke.log "$out"/bench_tree.json "$out"/sample_rate.txt "$out"/gpu_some.log
