#!/bin/bash
# Run on the GPU box (gpurun): every bench workload, the ncu launch list of the default bench command, and `ncu --set full`
# captures of all kernels.  Outputs land in gpurun_out/ and are summarised into profiles/ afterwards with
# tools/ncu_summary.py and tools/ncu_lines.py (bench JSONs are never taken under a profiler).
set -u
TAG=${1:-r2_final}
OUT=gpurun_out
mkdir -p $OUT
python bench.py > $OUT/${TAG}_bench_decode48.json 2> $OUT/${TAG}_bench_decode48.err || echo "bench decode48 failed"
tail -c 400 $OUT/${TAG}_bench_decode48.json; echo
for w in encode48 decode16 mixed roundtrip48 file48 file16; do
  python bench.py --workload $w --distinct 512 > $OUT/${TAG}_bench_$w.json 2> $OUT/${TAG}_bench_$w.err || echo "bench $w failed"
  tail -c 300 $OUT/${TAG}_bench_$w.json | head -c 300; echo
done
python bench.py --impl reference --steps 3 --warmup 1 > $OUT/${TAG}_bench_reference_decode48.json 2>/dev/null
ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $OUT/${TAG}_launches_decode48.csv \
    python bench.py --steps 2 --warmup 1 --no-cpu-baseline --no-secondary > $OUT/${TAG}_launches_decode48.log 2>&1
# one full step of the round trip = 8 encoder + 3 decoder kernels (no post-filter launch at 150 B).  bench.py brackets its first
# timed loop with cudaProfilerStart/Stop when LC3B_NCU_RANGE=1, so the captures hold steady-state launches only
LC3B_NCU_RANGE=1 ncu --set full --clock-control none --import-source on --profile-from-start off -c 11 -o $OUT/${TAG}_all \
    python bench.py --workload roundtrip48 --steps 1 --warmup 3 --quick --no-cpu-baseline --distinct 256 > $OUT/${TAG}_all.log 2>&1
# the decoder alone (inside a round trip its first kernel is billed for the write-back of what the encoder left dirty in L2)
LC3B_NCU_RANGE=1 ncu --set full --clock-control none --import-source on --profile-from-start off -c 3 -o $OUT/${TAG}_dec48 \
    python bench.py --steps 1 --warmup 3 --quick --no-cpu-baseline > $OUT/${TAG}_dec48.log 2>&1
# the small-batch path: BASELINE config 3 (16 384 streams): entropy, dequant_warp, tns_list, synth, ltpf
LC3B_NCU_RANGE=1 LC3B_GRAPH=0 ncu --set full --clock-control none --import-source on --profile-from-start off -c 5 -o $OUT/${TAG}_small \
    python bench.py --workload decode16 --streams 8192 --steps 2 --warmup 3 --quick --no-cpu-baseline > $OUT/${TAG}_small.log 2>&1
LC3B_NCU_RANGE=1 ncu --set full --clock-control none --import-source on --profile-from-start off -c 6 -o $OUT/${TAG}_multi \
    python bench.py --workload file48 --steps 2 --warmup 3 --no-cpu-baseline > $OUT/${TAG}_multi.log 2>&1
# summarise on the box and keep the reports out of gpurun_out (64 MiB limit for what travels back)
mkdir -p /tmp/ncu_reps
for r in all dec48 small multi; do
  if [ -f $OUT/${TAG}_$r.ncu-rep ]; then
    python tools/ncu_summary.py $OUT/${TAG}_$r.ncu-rep $OUT/${TAG}_${r}_ncu_summary.md $OUT/${TAG}_${r}_ncu_summary.json > /dev/null 2>&1 || echo "summary $r failed"
    : > $OUT/${TAG}_${r}_source_hotspots.txt
    for k in 0 1 2 3 4 5 6 7 8 9 10; do
      python tools/ncu_lines.py $OUT/${TAG}_$r.ncu-rep $k 12 >> $OUT/${TAG}_${r}_source_hotspots.txt 2>/dev/null && echo >> $OUT/${TAG}_${r}_source_hotspots.txt || break
    done
    mv $OUT/${TAG}_$r.ncu-rep /tmp/ncu_reps/
  fi
done
ls -la $OUT | tail -40
