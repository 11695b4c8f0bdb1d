#!/bin/bash
# compute-sanitizer over the kernel parity tests (memcheck, then racecheck); summaries -> gpurun_out/sanitizer_*.txt
# (copied to profiles/ by hand).  Each tool gets its own process per test file and a wall-clock limit.
mkdir -p gpurun_out
FILES=${FILES:-"tests/test_gpu_conv.py tests/test_gpu_preprocess.py tests/test_gpu_crops.py tests/test_gpu_detect_post.py tests/test_gpu_tracker.py tests/test_gpu_engine.py"}
for tool in ${TOOLS:-memcheck racecheck}; do
  out=gpurun_out/sanitizer_$tool.txt
  echo "# compute-sanitizer --tool $tool over the -m gpu parity tests ($(nvidia-smi --query-gpu=name --format=csv,noheader | head -1), $(compute-sanitizer --version | head -2 | tail -1))" > $out
  for f in $FILES; do
    log=gpurun_out/sanitizer_${tool}_$(basename $f .py).log
    timeout ${LIMIT:-420} compute-sanitizer --tool $tool --print-limit 20 --error-exitcode 86 \
      python -m pytest $f -q -m gpu -x -p no:cacheprovider ${PYTEST_ARGS} > $log 2>&1
    code=$?
    echo "$f: exit $code | $(grep -E '^=+ (ERROR|RACECHECK) SUMMARY' $log | tail -1) | $(grep -E ' passed| failed| error' $log | tail -1)" >> $out
    grep -E "^=+ (Invalid|Error|Race|Warning|Hazard)" $log | sort | uniq -c | sort -rn | head -8 >> $out
  done
done
cat gpurun_out/sanitizer_*.txt
