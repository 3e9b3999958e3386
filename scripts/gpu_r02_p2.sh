#!/bin/bash
# L2-sized conv passes (verdict item 3)
cd "$(dirname "$0")/.." || exit 1
mkdir -p gpurun_out; O=gpurun_out
echo "# bench.py --forward-only --steps 5 --warmup 3, 10 000 clips x 64 frames; key 3 = frames per conv pass" > $O/r02p2_table.txt
for t in ${VARIANTS:-"3=16384" "3=32768" "3=65536"}; do
  args=""; for kv in $t; do args="$args --tuning $kv"; done
  timeout 600 python bench.py --forward-only --steps 5 --warmup 3 $args > $O/r02p2.json 2> $O/r02p2.err; rc=$?
  python - <<PY >> $O/r02p2_table.txt
import json
for line in open("$O/r02p2.json"):
    if line.startswith("{"):
        d=json.loads(line); st=d.get("stage_ms_per_step",{})
        print("%-18s %7.2f ms/step  stem %6.2f  conv3 %5.2f  conv4 %5.2f" % ("$t", d["ms_per_step"], st.get("stem_fused",0), st.get("conv3_igemm",0), st.get("conv4_igemm_pool",0)))
PY
done
cat $O/r02p2_table.txt
