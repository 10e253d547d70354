#!/bin/bash
# One GPU run for the shared fit tail: the launch sequences and results of every entry point against a checkout of the
# parent commit at $1 (ab_results.py), the GPU suite, smoke, and bench.py's granule / tiles / shards / mosaic configs,
# alternating parent and change, twice each.  Everything lands in the output directory.
#   bash profiles/pipetail/run_gpu.sh <parent checkout with its library built> <output directory>
PARENT=$(cd "${1:?parent checkout}" && pwd)
mkdir -p "${2:?output directory}"
OUT=$(cd "$2" && pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/nvsmi.txt" 2>&1
nvidia-smi -L >> "$OUT/nvsmi.txt" 2>&1
{
  python profiles/pipetail/ab_results.py dump "$PARENT" "$OUT/results_parent.pt"
  python profiles/pipetail/ab_results.py dump . "$OUT/results_change.pt"
  python profiles/pipetail/ab_results.py compare "$OUT/results_parent.pt" "$OUT/results_change.pt"; echo "compare rc=$?"
} > "$OUT/ab.log" 2>&1
timeout 900 python -m pytest tests -m gpu -q -rs > "$OUT/pytest_gpu.log" 2>&1; echo "pytest rc=$?" | tee -a "$OUT/pytest_gpu.log"
timeout 300 python __graft_entry__.py smoke > "$OUT/smoke.log" 2>&1; echo "smoke rc=$?" | tee -a "$OUT/smoke.log"
for rep in 1 2; do
  for cfg in granule tiles shards mosaic; do
    for arm in parent change; do
      dir=$([ $arm = parent ] && echo "$PARENT" || pwd)
      (cd "$dir" && timeout 600 python bench.py --gpus 1 --config $cfg --steps 50 --warmup 5 --no-cpu) \
          > "$OUT/bench_${cfg}_${arm}_$rep.json" 2> "$OUT/bench_${cfg}_${arm}_$rep.err"
      echo "bench $cfg $arm $rep rc=$?"
    done
  done
done
