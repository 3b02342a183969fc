#!/bin/bash
# Measurements of the selection-pass / compaction-grid split (DESIGN.md §4.1, §5.2).
# usage: tools/r03_select_split.sh measure|final OUT_DIR   (OUT_DIR: where every result file is written)
#   measure: card, new many-rows test, output dumps of the parent build (tools/bin/libv_parent.so) and the new one
#            compared array by array, the alternating A/B (tools/ab_variants.py: in-tree library, parent, (U, CTAs/SM)
#            variants of the compaction grid), torch.profiler kernel tables;
#   final:   the GPU suite, smoke() and the default bench line.
# tools/bin/libv_parent.so is the parent commit's kvpress_b200/csrc built with kvpress_b200/build.py's nvcc flags;
# the variants are the in-tree objects with select_compact.cu rebuilt at other kCompactU / kCompactCtas values.
cd "$(dirname "$0")/.."
O=${2:?usage: $0 measure|final OUT_DIR}
mkdir -p "$O"
if [ "$1" = "measure" ]; then
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/card.txt 2>&1
timeout 300 python -m pytest -m gpu -q -p no:cacheprovider tests/test_gpu_many_rows.py > $O/many_rows.txt 2>&1
echo "many_rows rc=$?" >> $O/many_rows.txt

WLS="ea_128k knorm_128k snapkv_32k keydiff_128k rerotate_knorm_128k adakv_ea_128k"
for w in $WLS; do
  KVPRESS_B200_LIB=tools/bin/libv_parent.so timeout 200 python bench.py --workload $w --steps 2 --warmup 1 --no-cpu \
      --no-e2e --no-extras --dump-outputs $O/dump/parent/$w > $O/dump_parent_$w.json 2> $O/dump_parent_$w.err
  timeout 200 python bench.py --workload $w --steps 2 --warmup 1 --no-cpu --no-e2e --no-extras \
      --dump-outputs $O/dump/new/$w > $O/dump_new_$w.json 2> $O/dump_new_$w.err
done
python - "$O" $WLS > $O/dump_compare.txt 2>&1 <<'PY'
import os, sys
import numpy as np
out = sys.argv[1]
for w in sys.argv[2:]:
    a, b = os.path.join(out, "dump", "parent", w), os.path.join(out, "dump", "new", w)
    names = sorted(os.listdir(a)) if os.path.isdir(a) else []
    if not names:
        print(w, "NO DUMP"); continue
    for n in names:
        x, y = np.load(os.path.join(a, n)), np.load(os.path.join(b, n))
        print(f"{w:22s} {n:22s} {str(x.shape):22s} array_equal={np.array_equal(x, y)}")
PY
rm -rf $O/dump

AB_EXTRA=0 AB_WORKLOADS=ea_128k,knorm_128k,snapkv_32k,snapkv_128k_70b,keydiff_128k,rerotate_knorm_128k,adakv_ea_128k,decoding_knorm \
  timeout 600 python tools/ab_variants.py > $O/ab.txt 2>&1
timeout 300 python tools/kernel_table.py ea_128k knorm_128k streaming_128k > $O/kernels_new.txt 2>&1
KVPRESS_B200_LIB=tools/bin/libv_parent.so timeout 300 python tools/kernel_table.py ea_128k knorm_128k \
  > $O/kernels_parent.txt 2>&1
tail -n 3 $O/card.txt $O/many_rows.txt $O/dump_compare.txt $O/ab.txt
fi

if [ "$1" = "final" ]; then
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/card_final.txt 2>&1
timeout 600 python -m pytest -m gpu -q -p no:cacheprovider tests > $O/gpu_tests.txt 2>&1
echo "gpu tests rc=$?" >> $O/gpu_tests.txt
timeout 300 python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" > $O/smoke.txt 2>&1
timeout 600 python bench.py --gpus 1 > $O/bench_ea_128k.json 2> $O/bench_ea_128k.err
tail -n 3 $O/gpu_tests.txt $O/smoke.txt
fi
