#!/bin/bash
# Round 3c, GPU call 1: lit ground tiles (lit_tiles.h).  The card, then the same-box A/B of the parent library
# (tools/ab_build.sh parent "" <parent commit>) and this tree on all nine configs, the new GPU tests, the whole GPU suite,
# smoke(), and bench.py --dump-outputs with each library.  Everything is written under OUTPUT_DIR.
#   tools/gpu_calls/r3c_call01.sh OUTPUT_DIR
out=${1:?usage: r3c_call01.sh OUTPUT_DIR}
cd "$(dirname "$0")/../.."
mkdir -p "$out"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader > "$out"/card.txt 2>&1
cfgs="cfg5-repeat cfg5-moon cfg3-house cfg3-night-house cfg2-hollow-sphere cfg1-sample cfg4-bunny cfg4-bunny-d12 cfg4-bunny-full-d14"
timeout 900 python tools/ab_fast.py "$cfgs" "parent tree parent tree" 5 > "$out"/ab.txt 2>&1
timeout 600 python -m pytest -q -m gpu tests/test_gpu_lit_tiles.py > "$out"/gpu_lit.log 2>&1
timeout 900 python -m pytest -q -m gpu tests > "$out"/gpu_suite.log 2>&1
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > "$out"/smoke.log 2>&1; echo "smoke rc=$?" >> "$out"/smoke.log
timeout 600 python bench.py --gpus 1 --steps 5 --warmup 2 --dump-outputs "$out"/dump_tree > "$out"/bench_tree.json 2> "$out"/bench_tree.err
FTB_LIB=$PWD/ab/libftb_parent.so timeout 600 python bench.py --gpus 1 --steps 5 --warmup 2 --dump-outputs "$out"/dump_parent > "$out"/bench_parent.json 2> "$out"/bench_parent.err
OUT="$out" python - > "$out"/dump_compare.txt 2>&1 <<'PY'
import glob, os, numpy as np
for a in sorted(glob.glob(os.environ["OUT"] + "/dump_tree/*.npy")):
    b = a.replace("dump_tree", "dump_parent")
    x, y = np.load(a), np.load(b)
    print(os.path.basename(a), x.shape, "identical" if np.array_equal(x, y, equal_nan=True) else "DIFFERENT")
PY
rm -rf "$out"/dump_tree "$out"/dump_parent
tail -n 3 "$out"/ab.txt "$out"/gpu_lit.log "$out"/gpu_suite.log "$out"/smoke.log "$out"/dump_compare.txt
