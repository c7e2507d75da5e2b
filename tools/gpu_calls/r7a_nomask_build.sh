#!/bin/bash
# Builds ab/libftb_nomask.so, the "nomask" arm of tools/gpu_calls/r7a_call02.sh (profiles/r7a_tile_items_ab.txt section 2): the
# library of commit 057664b (the masks read by every FT_PAIRG / FT_CSGN variant) with the one line that hands the kernel the
# masks replaced by `F.tile_items = nullptr;`, so the kernels carry the masks' code but never receive any.
#   tools/gpu_calls/r7a_nomask_build.sh
set -e
root=$(cd "$(dirname "$0")/../.." && pwd)
work=$(mktemp -d /tmp/ftb_nomask_XXXXXX)
git -C "$root" archive 057664b functracer_b200/csrc include | tar -x -C "$work"
cd "$work/functracer_b200/csrc"
sed -i 's/F.tile_items = sizeof(R) == 4 \&\& pd->items_valid ? static_cast<const unsigned\*>(pd->items.p) : nullptr;/F.tile_items = nullptr;/' cuda/api.cu
grep -q "F.tile_items = nullptr;" cuda/api.cu
make cuda -j8 "F32_MATH=-use_fast_math -DFTB_FAST_MATH" > "$work/make.log" 2>&1 || { tail -20 "$work/make.log"; exit 1; }
mkdir -p "$root/ab" && cp "$work/functracer_b200/libfunctracer_b200.so" "$root/ab/libftb_nomask.so"
echo "-> ab/libftb_nomask.so"
rm -rf "$work"
