#!/usr/bin/env bash
# Qwen3 (QK-norm + decoupled head dim) on one B200: GPU suite, smoke, fused-kernel benchmark, step times, the GPT-2 headline
# A/B against the parent tree, memcheck.  The parent tree is a `git archive` of the previous commit under ab_tmp/base
# (git-ignored, built beforehand; see DEV_NOTES §1).  Results go to $OUT (default qwen3_out/).
#   bash scripts/gpu_qwen3.sh tests   (GPU suite, smoke, kernel benchmark)
#   bash scripts/gpu_qwen3.sh perf    (step times, QK-norm cost, headline A/B, memcheck)
set -uo pipefail
STAGE=${1:-tests}
OUT=${OUT:-qwen3_out}
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/card_$STAGE.txt

if [ $STAGE = tests ]; then
# 1. the whole GPU suite, then smoke()
timeout 2400 python -m pytest tests -q -m gpu -p no:cacheprovider > $OUT/pytest_gpu.txt 2>&1
echo "pytest gpu exit=$?" | tee -a $OUT/summary.txt
tail -5 $OUT/pytest_gpu.txt | tee -a $OUT/summary.txt
python -c "import __graft_entry__ as g; g.smoke()" > $OUT/smoke.txt 2>&1
echo "smoke exit=$?" | tee -a $OUT/summary.txt
if ! grep -q "pytest gpu exit=0" $OUT/summary.txt; then
  grep -E "^(FAILED|ERROR)" $OUT/pytest_gpu.txt | head -40
  exit 1
fi
# 2. fused-kernel benchmark at 1.7B shapes
timeout 600 python scripts/qk_norm_bench.py --out $OUT/qk_norm_bench.json > $OUT/qk_norm_bench.log 2>&1
echo "qk_norm_bench exit=$?" | tee -a $OUT/summary.txt
exit 0
fi

# 3. training steps (CUDA graph).  "qwen3-1.7b-noqk" is the 1.7B shape with qk_norm=False (plain RoPE): the cost of QK-norm.
step() {  # model batch seq
  timeout 900 python - "$1" "$2" "$3" <<'EOF' 2>&1 | tail -1
import dataclasses, runpy, sys
from distributedtraining_b200.models import transformer as t
t.PRESETS["qwen3-1.7b-noqk"] = dataclasses.replace(t.PRESETS["qwen3-1.7b"], name="qwen3-1.7b-noqk", qk_norm=False)
m, b, s = sys.argv[1:4]
sys.argv = ["step_bench.py", "--model", m, "--batch", b, "--seq", s, "--steps", "10", "--warmup", "3"]
runpy.run_path("scripts/step_bench.py", run_name="__main__")
EOF
}
for run in "qwen3-0.6b 8 512" "qwen3-0.6b 2 2048" "qwen3-1.7b 8 512" "qwen3-1.7b-noqk 8 512" "qwen3-1.7b 2 2048" \
           "qwen3-1.7b-noqk 2 2048" "qwen3-4b 2 2048"; do
  set -- $run
  r=$(step $1 $2 $3)
  case "$r" in \{*) ;; *) r="{\"model\": \"$1\", \"batch\": $2, \"seq\": $3, \"error\": \"$(echo $r | tr -d '"\\' | cut -c1-300)\"}" ;; esac
  echo "$r" | tee -a $OUT/step_qwen3.jsonl
done

# 4. GPT-2 headline, alternated with the parent tree
for i in 1 2 3; do
  for tree in base new; do
    dir=.; [ $tree = base ] && dir=ab_tmp/base
    r=$(cd $dir && timeout 600 python bench.py --gpus 1 2>/dev/null | tail -1)
    echo "{\"tree\": \"$tree\", \"run\": $i, \"result\": $r}" | tee -a $OUT/bench_headline_ab.jsonl
  done
done

# 5. memcheck over the Qwen3 GPU tests
timeout 1800 compute-sanitizer --tool memcheck --error-exitcode 9 python -m pytest tests/test_qwen3.py -q -m gpu \
    -p no:cacheprovider > $OUT/memcheck_qwen3.log 2>&1
echo "memcheck exit=$?" | tee -a $OUT/summary.txt
grep -E "ERROR SUMMARY|passed|failed" $OUT/memcheck_qwen3.log | tail -3 | tee -a $OUT/summary.txt
