#!/bin/bash
# Round 7a, GPU call 4: the masks in a second instance of the house-family variant (0x174b), launched only for frames whose masks pay.  The card, a clean build, a
# same-box A/B of the parent library and this tree on all nine configs, bench.py of the parent and this tree with
# --dump-outputs (frames compared bit for bit), the whole GPU suite and smoke().  Everything is written under OUTPUT_DIR.
#   tools/gpu_calls/r7a_call04.sh OUTPUT_DIR
out=${1:?usage: r7a_call04.sh OUTPUT_DIR}
cd "$(dirname "$0")/../.."
mkdir -p "$out"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader > "$out"/card.txt 2>&1
make -C functracer_b200/csrc clean > /dev/null 2>&1
timeout 900 python -c "import __graft_entry__ as g; g.build(verbose=False)" > "$out"/build.log 2>&1; echo "build rc=$?" >> "$out"/build.log
all="cfg5-repeat cfg3-house cfg3-night-house cfg5-moon cfg2-hollow-sphere cfg1-sample cfg4-bunny cfg4-bunny-d12 cfg4-bunny-full-d14"
timeout 1500 python tools/ab_fast.py "$all" "parent tree parent tree parent" 5 > "$out"/ab.txt 2>&1; echo "ab rc=$?" >> "$out"/ab.txt
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader >> "$out"/card.txt 2>&1
timeout 600 python bench.py --gpus 1 --steps 5 --warmup 2 --dump-outputs "$out"/dump_tree > "$out"/bench_tree.json 2> "$out"/bench_tree.err
FTB_LIB=$PWD/ab/libftb_parent.so timeout 600 python bench.py --gpus 1 --steps 5 --warmup 2 --dump-outputs "$out"/dump_parent > "$out"/bench_parent.json 2> "$out"/bench_parent.err
python - "$out" > "$out"/dumps_compare.txt 2>&1 <<'PY'
import glob, os, sys
import numpy as np
out = sys.argv[1]
names = sorted(os.path.basename(p) for p in glob.glob(os.path.join(out, "dump_parent", "*.npy")))
print("%d dumped frames" % len(names))
for n in names:
    a, b = np.load(os.path.join(out, "dump_parent", n)), np.load(os.path.join(out, "dump_tree", n))
    print("%-40s %s" % (n, "bit-identical" if a.shape == b.shape and a.tobytes() == b.tobytes() else "DIFFERENT"))
PY
timeout 2400 python -m pytest -q -m gpu -rs tests > "$out"/gpu_suite.log 2>&1; echo "gpu_suite rc=$?" >> "$out"/gpu_suite.log
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > "$out"/smoke.log 2>&1; echo "smoke rc=$?" >> "$out"/smoke.log
tail -n 3 "$out"/build.log "$out"/gpu_suite.log "$out"/smoke.log
cat "$out"/card.txt "$out"/ab.txt "$out"/dumps_compare.txt
