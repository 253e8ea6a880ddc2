#!/bin/bash
# round 3, call A (1 GPU): fused decode attention with the cached K/V loaded ahead of its grid-dependency wait (B200_ATTN_PREFETCH).
# The card, the whole GPU suite (incl. tests/test_gpu_attn_prefetch.py), the attention phase timeline in both orders, then the default
# bench line alternately with B200_ATTN_PREFETCH=0 and =1 (same binary), 3 runs each, then smoke().
OUT=$(realpath -m "${1:?usage: $0 OUTPUT_DIR}")
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/r03a_gpu.csv 2>&1; cat $OUT/r03a_gpu.csv
( timeout 1500 python -m pytest tests -q -m gpu -p no:cacheprovider ) > $OUT/r03a_gpu_suite.log 2>&1; echo "gpu suite rc=$?"; tail -4 $OUT/r03a_gpu_suite.log | cut -c1-300
for pf in 0 1; do
  B200_ATTN_PREFETCH=$pf timeout 300 python tools/decode_timeline.py > $OUT/r03a_attn_timeline_pf$pf.txt 2>&1; echo "timeline pf=$pf rc=$?"; tail -2 $OUT/r03a_attn_timeline_pf$pf.txt | cut -c1-300
done
for run in 1 2 3; do
  for pf in 0 1; do
    B200_ATTN_PREFETCH=$pf timeout 600 python bench.py > $OUT/r03a_bench_pf${pf}_run$run.json 2> $OUT/r03a_bench_pf${pf}_run$run.err; echo "bench pf=$pf run=$run rc=$?"
  done
done
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/r03a_smoke.log 2>&1; echo "smoke rc=$?"; tail -1 $OUT/r03a_smoke.log
OUT=$OUT python - <<'PY'
import os
import glob, json, statistics
for pf in (0, 1):
    ms, bits = [], []
    for f in sorted(glob.glob(os.environ["OUT"] + f"/r03a_bench_pf{pf}_run*.json")):
        try:
            d = json.loads(open(f).read().strip().splitlines()[-1])
            ms.append(d["ms_per_step"]); bits.append(d.get("cpu_baseline", {}).get("parity", {}).get("bit_identical"))
        except Exception as e:
            print(f, "ERR", e)
    if ms:
        print(f"B200_ATTN_PREFETCH={pf}: ms_per_step {[round(x, 4) for x in ms]} median {statistics.median(ms):.4f} spread {max(ms) - min(ms):.4f} bit_identical {bits}")
PY
