#!/bin/bash
# A/B of the resblock epilogue work: base library (build_variants/librvcb200_base.so, tools/build_variant.sh <rev> base)
# against the library in the tree.  Default bench line alternately, three times each; the dumped outputs of both, default
# precision and fp16, compared byte for byte; per-launch kernel times of one step (tools/launch_table.py) for both;
# then the GPU suite and smoke().  Everything it writes goes to the directory given as $1.
out=${1:?usage: tools/gpu_rbepi_ab.sh OUT_DIR}
mkdir -p "$out"
export AB_OUT=$out
export PYTHONUNBUFFERED=1
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm --format=csv | tee $out/gpu.csv
BASE=build_variants/librvcb200_base.so
run() {  # tag, lib ("" = in tree), bench args...
  local tag=$1 lib=$2; shift 2
  RVCB200_LIB=$lib timeout 400 python bench.py "$@" > $out/bench_$tag.json 2> $out/bench_$tag.err
  python - "$tag" <<'P'
import json, os, sys
d = json.load(open(f"{os.environ['AB_OUT']}/bench_{sys.argv[1]}.json"))
print(sys.argv[1], "ms", round(d["ms_per_step"], 3), "fp16 ms", round(d.get("fp16", {}).get("ms_per_step", 0), 3),
      "sm_mhz", d["clocks"].get("sm_mhz"), {k: round(x, 3) for k, x in d["time_by_class_ms_per_step"].items()},
      file=open(f"{os.environ['AB_OUT']}/bench_{sys.argv[1]}.summary", "w"))
P
}
for r in 1 2 3; do
  db=(); dh=()
  if [ $r = 1 ]; then db=(--dump-outputs $out/dump_base_default); dh=(--dump-outputs $out/dump_head_default); fi
  run base_$r $BASE --no-cpu-baseline --no-gpu-incumbent "${db[@]}"
  run head_$r "" --no-cpu-baseline --no-gpu-incumbent "${dh[@]}"
done
for v in base head; do
  lib=""; [ $v = base ] && lib=$BASE
  run ${v}_fp16dump "$lib" --precision fp16 --no-cpu-baseline --no-gpu-incumbent --no-parity --no-front-end \
    --dump-outputs $out/dump_${v}_fp16
done
for p in default fp16; do
  for f in $out/dump_base_$p/*; do
    cmp -s "$f" "$out/dump_head_$p/$(basename $f)" && echo "same $p $(basename $f)" || echo "DIFFERENT $p $(basename $f)"
  done
done | tee $out/dump_cmp.txt
rm -rf $out/dump_*_default $out/dump_*_fp16     # up to 64 MB each
RVCB200_LIB=$BASE timeout 400 python tools/launch_table.py --out $out/launches_base.json
timeout 400 python tools/launch_table.py --out $out/launches_head.json
python tools/launch_table.py --compare $out/launches_base.json $out/launches_head.json --filter rbconv_tc_kernel \
  | tee $out/rbconv_launches.md
cat $out/gpu.csv; grep -h . $out/bench_*.summary
# then the whole GPU suite and smoke() on the library in the tree
timeout 1200 python -m pytest tests -m gpu -q > $out/pytest_gpu.log 2>&1; tail -5 $out/pytest_gpu.log
timeout 600 python __graft_entry__.py smoke > $out/smoke.log 2>&1; echo "smoke rc $?"; tail -6 $out/smoke.log
