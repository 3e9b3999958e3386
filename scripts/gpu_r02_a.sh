#!/bin/bash
# Round-2 GPU session A: parity suite, A/B of the forward scheduling knobs, full bench line.
cd "$(dirname "$0")/.." || exit 1
mkdir -p gpurun_out
O=gpurun_out
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.limit --format=csv > $O/r02a_smi.txt 2>&1
timeout 1500 python -m pytest tests -m gpu -x -q > $O/r02a_gputests.log 2>&1; echo "pytest exit $?" >> $O/r02a_gputests.log
tail -5 $O/r02a_gputests.log
ab() { name=$1; shift; timeout 300 python bench.py --forward-only --steps 5 --warmup 3 "$@" > $O/r02a_ab_$name.json 2> $O/r02a_ab_$name.err; echo "$name exit $?"; python - <<PY
import json
try:
    d=json.loads(open("$O/r02a_ab_$name.json").read().strip().splitlines()[-1])
    print("$name", round(d["value"]), "videos/s", round(d["ms_per_step"],2), "ms/step; profiled", round(d["roofline"]["profiled_ms_per_step"],2), "sum", round(d["roofline"]["sum_of_stages_ms"],2), d["clocks"])
except Exception as e:
    print("$name: no line", e)
PY
}
ab old      --pipelines 1 --frames-per-pass 1048576
ab p2_128k  --pipelines 2 --frames-per-pass 131072
ab p2_64k   --pipelines 2 --frames-per-pass 65536
ab p3_64k   --pipelines 3 --frames-per-pass 65536
timeout 900 python bench.py --steps 10 --warmup 3 > $O/r02a_bench_n1.json 2> $O/r02a_bench_n1.err; echo "bench exit $?"
tail -c 3000 $O/r02a_bench_n1.json
