#!/bin/bash
set -u
OUT=gpurun_out; mkdir -p $OUT; T=${1:-r2_e}
timeout 900 python -m pytest tests/test_decoder_gpu.py tests/test_clip200_gpu.py tests/test_multi_frame_gpu.py -m gpu -q -x > $OUT/${T}_pytest.log 2>&1; echo "pytest rc=$?"; tail -4 $OUT/${T}_pytest.log
LC3B_DEQUANT=warp python bench.py --steps 100 --quick 2>/dev/null | sed 's/^/decode48 warp-dequant: /'
for s in 2048 8192 16384 32768; do
  for m in warp thread; do
    LC3B_DEQUANT=$m python bench.py --workload decode16 --streams $s --quick --steps 200 2>/dev/null | sed "s/^/decode16 streams=$s dequant=$m: /"
  done
done
ncu --metrics gpu__time_duration.sum --clock-control none -c 2000 --csv --log-file $OUT/${T}_launches_decode16.csv \
    python bench.py --workload decode16 --quick --steps 3 --warmup 3 > /dev/null 2>&1
python - <<PY
import csv
rows = [r for r in csv.reader(open("$OUT/${T}_launches_decode16.csv")) if len(r) > 5 and r[0].isdigit()]
names = [r[4] for r in rows]
idx = max(i for i, n in enumerate(names) if "entropy" in n)
for r in rows[idx:idx + 6]:
    print("   %-60s grid %-14s %8.1f us" % (r[4][:60], r[8], float(r[-1].replace(",", "")) / 1e3))
PY
