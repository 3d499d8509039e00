#!/bin/bash
# Round-end refresh after a change to the large-crowd path only (under gpurun, ONE GPU): GPU tests, smoke, the bench lines that
# carry large-crowd figures, the launch list of the default bench command, one full capture of the pair kernel, and
# compute-sanitizer over the large-crowd tests.  tools/merge_lines.py folds the lines into profiles/<round>_bench_lines.jsonl.
R=${1:-r02}
O=gpurun_out
python -m pytest tests -m gpu -q --tb=short 2>&1 | tail -3 > $O/final_gpu_tests.log
python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" > $O/final_smoke.log 2>&1
: > $O/${R}_large_lines.jsonl
python bench.py 2>$O/bench_err_default.log | tail -1 >> $O/${R}_large_lines.jsonl
python bench.py --dtype f32 --no-cpu-baseline 2>/dev/null | tail -1 >> $O/${R}_large_lines.jsonl
for dt in f64 f32; do
  python bench.py --workload 65536_hsfm_single_crowd --dtype $dt --no-cpu-baseline 2>/dev/null | tail -1 >> $O/${R}_large_lines.jsonl
done
ncu --metrics gpu__time_duration.sum --clock-control none -c 900 --csv --log-file $O/${R}_launches_bench.csv python bench.py --steps 20 --warmup 3 --no-cpu-baseline > $O/${R}_bench_under_ncu.log 2>&1
name=k_large_pairs_f64
SNP_BENCH_NO_LARGE=1 ncu --set full --clock-control none --import-source on -k regex:k_large_pairs -s 6 -c 1 -f -o $O/${R}_${name} python bench.py --workload 65536_hsfm_single_crowd --steps 3 --warmup 3 > /dev/null 2>&1
ncu -i $O/${R}_${name}.ncu-rep --page raw --csv > $O/${R}_${name}.raw.csv 2>/dev/null
ncu -i $O/${R}_${name}.ncu-rep --page source --csv --print-source sass > $O/${R}_${name}.source.csv 2>/dev/null
if [ $(stat -c %s $O/${R}_${name}.ncu-rep) -gt 8000000 ]; then rm -f $O/${R}_${name}.ncu-rep; fi
S=/usr/local/cuda/bin/compute-sanitizer
: > $O/${R}_sanitizer_large.txt
for tool in memcheck racecheck synccheck; do
  echo "=== $tool: large crowd (cull kernel, work list, persistent pair CTAs, list-walking finish; culled static grid of an unaligned slice; all pairs)" >> $O/${R}_sanitizer_large.txt
  timeout 170 $S --tool $tool --error-exitcode 9 python -m pytest -q -m gpu -x "tests/test_gpu_sizes_large.py::test_large_crowd_chunked_sums_and_exact_culling" "tests/test_gpu_sizes_large.py::test_large_crowd_tiled_kernel_vs_oracle" 2>&1 | grep -E "ERROR SUMMARY|RACECHECK SUMMARY|passed|failed|Error|error" | tail -4 >> $O/${R}_sanitizer_large.txt
done
cat $O/final_gpu_tests.log $O/final_smoke.log $O/${R}_sanitizer_large.txt; wc -l $O/${R}_large_lines.jsonl
