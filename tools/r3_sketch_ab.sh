#!/bin/sh
# c2 with and without the fp32 projection sketch on one GPU, alternating, 3 runs each, plus the sketch's own tests and counters.
#     sh tools/r3_sketch_ab.sh OUT_DIR
OUT=${1:?usage: sh tools/r3_sketch_ab.sh OUT_DIR}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/gpu.csv" 2>&1
python -m pytest -q -m gpu tests/test_f32_sketch.py > "$OUT/test_f32_sketch.log" 2>&1
echo "test_f32_sketch rc=$?"
python tools/sketch_stats.py > "$OUT/sketch_stats.log" 2>&1
echo "sketch_stats rc=$?"
for i in 1 2 3; do
  JV_F32_SKETCH=0 python bench.py --gpus 1 --steps 20 --warmup 3 --workload c2 --dump-outputs "$OUT/dump_off$i" > "$OUT/c2_off$i.json" 2> "$OUT/c2_off$i.err"
  echo "off$i rc=$?"
  JV_F32_SKETCH=1 python bench.py --gpus 1 --steps 20 --warmup 3 --workload c2 --dump-outputs "$OUT/dump_on$i" > "$OUT/c2_on$i.json" 2> "$OUT/c2_on$i.err"
  echo "on$i rc=$?"
done
python - "$OUT" <<'PY'
import json, sys, os
out = sys.argv[1]
for tag in ("off", "on"):
    for i in (1, 2, 3):
        try:
            d = json.loads(open(os.path.join(out, "c2_%s%d.json" % (tag, i))).read().strip().splitlines()[-1])
            print(tag, i, "value %.0f" % d["value"], "ms %.3f" % d["ms_per_step"], "recall", d["recall_at_10"], "parity", d["parity"]["ok"], "clocks", d.get("clocks_timed_region"))
        except Exception as e:
            print(tag, i, "ERR", e)
PY
