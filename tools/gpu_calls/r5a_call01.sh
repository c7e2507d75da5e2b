#!/bin/bash
# Round 5a, GPU call 1: path queries (ftb_trace_paths).  The card, the build, the new GPU tests, smoke(), bench.py with this tree
# and with the parent library (ab/libftb_parent.so, tools/ab_build.sh parent "" <parent commit>; --dump-outputs compared),
# tools/path_rate.py, the new GPU tests against four libraries with one planted mistake each (ab/libftb_plant_*.so: paths.cu
# with the weight not multiplied by L, the sample keys ignored, the FP32 planar self-skip dropped on bounce rays, the shadow-ray
# origin not offset), then the whole GPU suite.  Everything is written under OUTPUT_DIR.
#   tools/gpu_calls/r5a_call01.sh OUTPUT_DIR
out=${1:?usage: r5a_call01.sh OUTPUT_DIR}
cd "$(dirname "$0")/../.."
mkdir -p "$out"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader > "$out"/card.txt 2>&1
timeout 300 python -c "import __graft_entry__ as g; g.build(verbose=False)" > "$out"/build.log 2>&1; echo "build rc=$?" >> "$out"/build.log
timeout 1500 python -m pytest -q -m gpu -rs -s tests/test_gpu_path_queries.py > "$out"/gpu_paths.log 2>&1; echo "gpu_paths rc=$?" >> "$out"/gpu_paths.log
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > "$out"/smoke.log 2>&1; echo "smoke rc=$?" >> "$out"/smoke.log
timeout 600 python bench.py --gpus 1 --steps 5 --warmup 2 --dump-outputs "$out"/dump_tree > "$out"/bench_tree.json 2> "$out"/bench_tree.err
FTB_LIB=$PWD/ab/libftb_parent.so timeout 600 python bench.py --gpus 1 --steps 5 --warmup 2 --dump-outputs "$out"/dump_parent > "$out"/bench_parent.json 2> "$out"/bench_parent.err
timeout 600 python bench.py --gpus 1 --steps 5 --warmup 2 > "$out"/bench_tree2.json 2> "$out"/bench_tree2.err
OUT="$out" python - > "$out"/dump_compare.txt 2>&1 <<'PY'
import glob, os, numpy as np
for a in sorted(glob.glob(os.environ["OUT"] + "/dump_tree/*.npy")):
    b = a.replace("dump_tree", "dump_parent")
    x, y = np.load(a), np.load(b)
    print(os.path.basename(a), x.shape, "identical" if np.array_equal(x, y, equal_nan=True) else "DIFFERENT")
PY
rm -rf "$out"/dump_tree "$out"/dump_parent
timeout 600 python tools/path_rate.py > "$out"/path_rate.txt 2>&1
for plant in "weight_no_L fp64_paths_are" "shadow_no_offset fp64_paths_are" "keys_ignored sample_keys" "no_bounce_skip fp32"; do
  set -- $plant
  FTB_LIB=$PWD/ab/libftb_plant_$1.so timeout 600 python -m pytest -q -m gpu -x -k "$2" tests/test_gpu_path_queries.py > "$out"/plant_$1.log 2>&1
  echo "plant $1 (-k $2) rc=$?" >> "$out"/plants.txt
done
timeout 2400 python -m pytest -q -m gpu tests --ignore=tests/test_gpu_path_queries.py > "$out"/gpu_suite.log 2>&1; echo "gpu_suite rc=$?" >> "$out"/gpu_suite.log
tail -n 3 "$out"/build.log "$out"/gpu_paths.log "$out"/smoke.log "$out"/dump_compare.txt "$out"/path_rate.txt "$out"/plants.txt "$out"/gpu_suite.log
