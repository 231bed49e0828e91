#!/usr/bin/env bash
# Head-dim-128 attention on one B200: GPU suite, smoke, kernel benchmark, step and headline A/B against the parent tree,
# memcheck.  The parent tree is a `git archive` of the previous commit under ab_tmp/base (git-ignored, built beforehand; see
# DEV_NOTES §1).  Results go to $OUT (default hd128_out/).
#   bash scripts/gpu_hd128.sh tests   (GPU suite, smoke, kernel benchmark)
#   bash scripts/gpu_hd128.sh ab      (step and headline A/B, memcheck)
set -uo pipefail
STAGE=${1:-tests}
OUT=${OUT:-hd128_out}
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/card.txt

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

# 2. kernel benchmark
timeout 1200 python scripts/attn_bench.py --out $OUT/attn_hd128_bench.json > $OUT/attn_bench.log 2>&1
echo "attn_bench exit=$?" | tee -a $OUT/summary.txt
exit 0
fi

# 3. llama-3.2-3b step: this tree vs the parent (hd 128 attention = fp32 reference there).  The parent has no 3B preset:
#    the same shape is registered before step_bench runs.
step() {  # tree batch seq [--no-graph]
  local dir=.; [ $1 = base ] && dir=ab_tmp/base
  (cd $dir && timeout 900 python - "$2" "$3" "${4:-}" <<'EOF' 2>&1 | tail -1
import runpy, sys
from distributedtraining_b200.models import transformer as t
t.PRESETS.setdefault("llama-3.2-3b", t.ModelConfig(family="llama", name="llama-3.2-3b", vocab_size=128256, n_positions=131072,
                     n_embd=3072, n_layer=28, n_head=24, n_kv_head=8, ffn=8192, eps=1e-5, rope_theta=500000.0))
b, s, ng = sys.argv[1:4]
sys.argv = ["step_bench.py", "--model", "llama-3.2-3b", "--batch", b, "--seq", s, "--steps", "10", "--warmup", "3"] + ([ng] if ng else [])
runpy.run_path("scripts/step_bench.py", run_name="__main__")
EOF
  )
}
for shape in "8 512" "2 2048"; do
  set -- $shape
  ng=""
  r=$(step base $1 $2)
  case "$r" in \{*) ;; *) echo "base $shape graph: $r" >> $OUT/step_errors.txt; ng=--no-graph; r=$(step base $1 $2 $ng) ;; esac
  echo "{\"tree\": \"base\", \"result\": $r}" | tee -a $OUT/step_llama3b_ab.jsonl
  r=$(step new $1 $2 $ng)
  echo "{\"tree\": \"new\", \"result\": $r}" | tee -a $OUT/step_llama3b_ab.jsonl
  [ -n "$ng" ] && { r=$(step new $1 $2); echo "{\"tree\": \"new\", \"result\": $r}" | tee -a $OUT/step_llama3b_ab.jsonl; }
done

# 4. GPT-2 headline (hd 64), alternated
for i in 1 2 3; do
  for tree in base new; do
    dir=.; [ $tree = base ] && dir=ab_tmp/base
    r=$(cd $dir && timeout 600 python bench.py --gpus 1 2>/dev/null | tail -1)
    echo "{\"tree\": \"$tree\", \"run\": $i, \"result\": $r}" | tee -a $OUT/bench_headline_ab.jsonl
  done
done

# 5. memcheck over the new attention tests
timeout 1800 compute-sanitizer --tool memcheck --error-exitcode 9 python -m pytest tests/test_attention_hd128_gpu.py -q \
    -p no:cacheprovider > $OUT/memcheck_hd128.log 2>&1
echo "memcheck exit=$?" | tee -a $OUT/summary.txt
grep -E "ERROR SUMMARY|passed|failed" $OUT/memcheck_hd128.log | tail -3 | tee -a $OUT/summary.txt
