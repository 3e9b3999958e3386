#!/bin/bash
cd "$(dirname "$0")/.." || exit 1
mkdir -p gpurun_out; O=gpurun_out
timeout 1500 python -m pytest tests -m gpu -x -q > $O/r02i_gputests.log 2>&1; echo "pytest exit $?" >> $O/r02i_gputests.log; tail -4 $O/r02i_gputests.log
ab() { name=$1; shift; timeout 300 python bench.py --forward-only --steps 5 --warmup 3 "$@" > $O/r02i_ab_$name.json 2> $O/r02i_ab_$name.err; echo "$name exit $?"; python - <<PY
import json
try:
    d=json.loads(open("$O/r02i_ab_$name.json").read().strip().splitlines()[-1])
    st=d["stage_ms_per_step"]
    print("$name", round(d["value"]), "videos/s", round(d["ms_per_step"],2), "ms/step;", {k: round(v,2) for k,v in st.items()})
except Exception as e:
    print("$name: no line", e)
PY
}
ab base
