#!/bin/bash
# One B200: the round's final evidence pass.  Tests, bench lines of every single-GPU config, the reference arm, the mask-side
# benches with SciPy beside them, the ncu launch list of the bench command and full captures of the main kernels.
set -x
OUT=${OUT:-out}  # output directory (git-ignored)
mkdir -p "$OUT"
timeout 900 python -m pytest tests -m gpu -q 2>&1 | tail -6 > $OUT/pytest_gpu.txt
cat $OUT/pytest_gpu.txt
timeout 600 python bench.py > $OUT/bench_c3.json 2> $OUT/bench_c3.err
cat $OUT/bench_c3.json; tail -n 3 $OUT/bench_c3.err
timeout 300 python bench.py --impl reference --steps 2 --warmup 1 > $OUT/bench_ref.json 2> $OUT/bench_ref.err
cat $OUT/bench_ref.json
for w in c1 c2 c4; do
  timeout 300 python bench.py --workload $w --steps 3 --warmup 3 > $OUT/bench_$w.json 2> $OUT/bench_$w.err
  head -c 400 $OUT/bench_$w.json; echo; tail -n 2 $OUT/bench_$w.err
done
timeout 300 python bench.py --workload c5 --scaling weak --steps 3 --warmup 3 > $OUT/bench_c5_weak1.json 2> $OUT/bench_c5_weak1.err
head -c 400 $OUT/bench_c5_weak1.json; echo; tail -n 2 $OUT/bench_c5_weak1.err
timeout 300 python scripts/bench_continuous.py > $OUT/bench_continuous.json 2> $OUT/bench_continuous.err
cat $OUT/bench_continuous.json
timeout 600 python scripts/bench_mask.py --cpu > $OUT/bench_mask_c2.json 2> $OUT/bench_mask_c2.err
cat $OUT/bench_mask_c2.json; tail -n 3 $OUT/bench_mask_c2.err
timeout 300 python scripts/bench_mask.py --shape 640x880x880 --reps 3 > $OUT/bench_mask_c3.json 2> $OUT/bench_mask_c3.err
cat $OUT/bench_mask_c3.json
# ncu: launch list of the bench command itself, then full captures
timeout 500 ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file $OUT/launches_bench.csv \
    python bench.py --steps 1 --warmup 1 > $OUT/bench_under_ncu.json 2> $OUT/bench_under_ncu.err
timeout 300 ncu --set full --clock-control none --import-source on -k regex:k_sweep_dense -s 6 -c 2 -f -o $OUT/final_sweep_dense \
    python scripts/profile_step.py --workload c3 --intensity f64_dense --iters 12 > $OUT/ncu1.log 2>&1
timeout 300 ncu --set full --clock-control none --import-source on -k regex:k_init_hist_shared -c 1 -f -o $OUT/final_init_hist \
    python scripts/profile_step.py --workload c3 --intensity f64_dense --iters 2 > $OUT/ncu2.log 2>&1
timeout 300 ncu --set full --clock-control none --import-source on -k regex:k_cancel -s 40 -c 1 -f -o $OUT/final_cancel \
    python scripts/profile_step.py --workload c3 --intensity f64_dense --iters 50 > $OUT/ncu3.log 2>&1
timeout 300 ncu --set full --clock-control none --import-source on -k "regex:k_edt_lines|k_cc_merge" -c 4 -f -o $OUT/final_mask \
    python scripts/bench_mask.py --shape 640x880x880 --reps 1 > $OUT/ncu4.log 2>&1
ls -la $OUT | tail -12
