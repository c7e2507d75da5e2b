#!/bin/bash
# Builds an A/B copy of libfunctracer_b200.so into ab/ (git-ignored, but shipped to the GPU box by gpurun).
#   tools/ab_build.sh NAME ["extra nvcc flags for the FP32 kernels"] [GIT_REV]
# With GIT_REV the library is built from that commit's sources, else from the working tree.  The copy is selected
# at run time with FTB_LIB=$PWD/ab/libftb_NAME.so (functracer_b200/api.py); see tools/ab_bench.sh.
# AB_MAKE_ARGS in the environment is appended to the make command line (through eval, e.g. AB_MAKE_ARGS="EXTRA=-DFTB_UNIT_CAP=128 'F32_FEATS=0xfff 0x74b'").
# Prints the SASS size and the spill summary of every FP32 variant, the numbers to look at before spending GPU time.
set -e
name=$1; flags=$2; rev=$3
root=$(cd "$(dirname "$0")/.." && pwd)
work=$(mktemp -d /tmp/ftb_ab_XXXXXX)
if [ -n "$rev" ]; then git -C "$root" archive "$rev" functracer_b200/csrc include | tar -x -C "$work"
else mkdir -p "$work/functracer_b200" && cp -r "$root/functracer_b200/csrc" "$work/functracer_b200/" && cp -r "$root/include" "$work/"; fi
cd "$work/functracer_b200/csrc" && rm -rf build
eval make cuda -j8 "'F32_MATH=-use_fast_math -DFTB_FAST_MATH $flags'" $AB_MAKE_ARGS > "$work/make.log" 2>&1 || { tail -20 "$work/make.log"; exit 1; }
mkdir -p "$root/ab" && cp "$work/functracer_b200/libfunctracer_b200.so" "$root/ab/libftb_$name.so"
for f in build/render_f32_*.o; do
  n=$(cuobjdump -sass "$f" | awk '/Function :/{k=$3} /^ +\/\*[0-9a-f]+\*\/ /{c[k]++} END{for(k in c) if (k ~ /Lb0/) print c[k]}')
  s=$(grep -A2 'render_kernelIf.*Lb0' "${f%.o}.ptxas.log" | grep -o '[0-9]* bytes stack frame, [0-9]* bytes spill stores, [0-9]* bytes spill loads' | head -1)
  echo "$(basename "$f" .o): $n SASS instructions; $s"
done
echo "-> ab/libftb_$name.so"
rm -rf "$work"
