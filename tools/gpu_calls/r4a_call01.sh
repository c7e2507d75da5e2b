#!/bin/bash
# Round 4a, GPU call 1: crossing queries (ftb_intersect_all_rays).  The card, the new GPU tests, smoke(), bench.py with this tree
# and with the parent library (ab/libftb_parent.so, tools/ab_build.sh parent "" <parent commit>; --dump-outputs compared),
# tools/crossings_rate.py, then the whole GPU suite.  Everything is written under OUTPUT_DIR.
#   tools/gpu_calls/r4a_call01.sh OUTPUT_DIR
out=${1:?usage: r4a_call01.sh OUTPUT_DIR}
cd "$(dirname "$0")/../.."
mkdir -p "$out"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader > "$out"/card.txt 2>&1
timeout 300 python -c "import __graft_entry__ as g; g.build(verbose=False)" > "$out"/build.log 2>&1; echo "build rc=$?" >> "$out"/build.log
timeout 1200 python -m pytest -q -m gpu -rs -s tests/test_gpu_ray_crossings.py > "$out"/gpu_crossings.log 2>&1
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
timeout 600 python tools/crossings_rate.py > "$out"/crossings_rate.txt 2>&1
timeout 1200 python -m pytest -q -m gpu tests --ignore=tests/test_gpu_ray_crossings.py > "$out"/gpu_suite.log 2>&1
tail -n 3 "$out"/build.log "$out"/gpu_crossings.log "$out"/smoke.log "$out"/dump_compare.txt "$out"/crossings_rate.txt "$out"/gpu_suite.log
