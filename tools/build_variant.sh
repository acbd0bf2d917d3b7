#!/bin/bash
# Build build_variants/librvcb200_<tag>.so from comfy_rvc_b200/csrc/ and include/ of git rev $1 (or "wt" = working tree),
# with the flags of comfy_rvc_b200/build.py.  Select a variant at run time with RVCB200_LIB=<path>.
set -e
rev=$1; tag=${2:-$1}
root=$(cd "$(dirname "$0")/.." && pwd)
tmp=$(mktemp -d)
trap 'rm -rf $tmp' EXIT
mkdir -p $tmp/comfy_rvc_b200/csrc $tmp/include $root/build_variants
if [ "$rev" = "wt" ]; then
  cp $root/comfy_rvc_b200/csrc/*.cu $root/comfy_rvc_b200/csrc/*.cuh $tmp/comfy_rvc_b200/csrc/
  cp $root/include/rvcb200.h $tmp/include/
else
  git -C $root archive $rev comfy_rvc_b200/csrc include | tar -x -C $tmp
fi
flags=$(python3 -c "import sys; sys.path.insert(0, '$root/comfy_rvc_b200'); import build; print(' '.join(build.NVCC_FLAGS))")
objs=""
for f in $tmp/comfy_rvc_b200/csrc/*.cu; do
  o=${f%.cu}.o; objs="$objs $o"
  nvcc $flags -c $f -o $o &
done
for job in $(jobs -p); do wait $job; done
nvcc -shared -o $root/build_variants/librvcb200_$tag.so $objs -cudart static -Xcompiler -fPIC -gencode arch=compute_100a,code=sm_100a
echo built build_variants/librvcb200_$tag.so
