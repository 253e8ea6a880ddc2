#!/bin/bash
# round 3, call C (1 GPU): the default bench line of the parent commit against this tree in both attention orders, alternating, 3 runs each,
# plus the parent's per-launch timeline.  Set up before the call (tools/ab/ is not tracked):
#   mkdir -p tools/ab/parent && git archive <parent> | tar -x -C tools/ab/parent && make -C tools/ab/parent/llm_b200/csrc -j16 && make -C tools/ab/parent/oracle liboracle.so
OUT=$(realpath -m "${1:?usage: $0 OUTPUT_DIR}")
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/r03c_gpu.csv 2>&1; cat $OUT/r03c_gpu.csv
( cd tools/ab/parent && timeout 300 python tools/decode_timeline.py > $OUT/r03c_timeline_parent.txt 2>&1 ); echo "parent timeline rc=$?"; sed -n 5p $OUT/r03c_timeline_parent.txt
for run in 1 2 3; do
  ( cd tools/ab/parent && timeout 600 python bench.py > $OUT/r03c_bench_parent_run$run.json 2> $OUT/r03c_bench_parent_run$run.err ); echo "bench parent run=$run rc=$?"
  for pf in 0 1; do
    B200_ATTN_PREFETCH=$pf timeout 600 python bench.py > $OUT/r03c_bench_pf${pf}_run$run.json 2> $OUT/r03c_bench_pf${pf}_run$run.err; echo "bench pf=$pf run=$run rc=$?"
  done
done
OUT=$OUT python - <<'PY'
import os
import glob, json, statistics
for arm in ("parent", "pf0", "pf1"):
    ms, bits = [], []
    for f in sorted(glob.glob(os.environ["OUT"] + f"/r03c_bench_{arm}_run*.json")):
        try:
            d = json.loads(open(f).read().strip().splitlines()[-1])
            ms.append(d["ms_per_step"]); bits.append(d.get("cpu_baseline", {}).get("parity", {}).get("bit_identical"))
        except Exception as e:
            print(f, "ERR", e)
    if ms:
        print(f"{arm}: ms_per_step {[round(x, 4) for x in ms]} median {statistics.median(ms):.4f} spread {max(ms) - min(ms):.4f} bit_identical {bits}")
PY
