#!/bin/bash
# Round 4 measurements of the barrier-free dictionary insert (profiles/r04_*), written to OUTDIR.  PARENT is
# a built checkout of the parent commit (the "before" arm).
#   tools/_r04_dedup_ab.sh OUTDIR PARENT ab      stage times of both builds, alternated, on the bench
#                                                workload and on 8 GB of random text; kernel profiles
#   tools/_r04_dedup_ab.sh OUTDIR PARENT check   the new tests, smoke(), the whole GPU suite
#   tools/_r04_dedup_ab.sh OUTDIR PARENT bench   bench.py of both builds, outputs dumped and compared
#   tools/_r04_dedup_ab.sh OUTDIR PARENT full    tools/fullsize_check.py --config all
set -u
USAGE="usage: _r04_dedup_ab.sh OUTDIR PARENT ab|check|bench|full"
OUT=${1:?$USAGE}
PARENT=${2:?$USAGE}
WHAT=${3:?$USAGE}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv | tee "$OUT/r04_card.txt"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/r04_build.log" 2>&1 || { tail -30 "$OUT/r04_build.log"; exit 1; }
(cd "$PARENT" && python -c "import __graft_entry__ as g; g.build()") > "$OUT/r04_build_parent.log" 2>&1 || { tail -30 "$OUT/r04_build_parent.log"; exit 1; }
if [ "$WHAT" = ab ]; then
  for round in 1 2 3; do
    for arm in parent new; do
      root=.; [ $arm = parent ] && root=$PARENT
      timeout 300 python tools/dedup_ab.py --root "$root" --label $arm --steps 4 --warmup 2 2>>"$OUT/r04_stderr.log" | tail -1 | tee -a "$OUT/r04_dedup_ab_bench.jsonl"
    done
  done
  for arm in parent new; do
    root=.; [ $arm = parent ] && root=$PARENT
    timeout 300 python tools/dedup_ab.py --root "$root" --label $arm --steps 1 --warmup 1 \
        --profile "$OUT/r04_kernels_$arm.txt" 2>>"$OUT/r04_stderr.log" > /dev/null
  done
  for round in 1 2; do
    for arm in parent new; do
      root=.; [ $arm = parent ] && root=$PARENT
      timeout 400 python tools/dedup_ab.py --root "$root" --label $arm --workload random --steps 3 --warmup 1 \
          2>>"$OUT/r04_stderr.log" | tail -1 | tee -a "$OUT/r04_dedup_ab_random8GB.jsonl"
    done
  done
  for arm in parent new; do
    root=.; [ $arm = parent ] && root=$PARENT
    timeout 400 python tools/dedup_ab.py --root "$root" --label $arm --workload random --steps 1 --warmup 1 \
        --profile "$OUT/r04_kernels_random8GB_$arm.txt" 2>>"$OUT/r04_stderr.log" > /dev/null
  done
  python tools/dedup_ab.py --summarize "$OUT/r04_dedup_ab_bench.jsonl" "$OUT/r04_dedup_ab_random8GB.jsonl" | tee "$OUT/r04_dedup_ab_summary.txt"
elif [ "$WHAT" = check ]; then
  timeout 600 python -m pytest -q tests/test_dedup_slots_gpu.py 2>&1 | tee "$OUT/r04_pytest_dedup_slots.log" | tail -15
  timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tee "$OUT/r04_smoke.log" | tail -3
  timeout 900 python -m pytest -q -m gpu tests 2>&1 | tee "$OUT/r04_pytest_gpu.log" | tail -15
elif [ "$WHAT" = bench ]; then
  for arm in parent new; do
    root=.; [ $arm = parent ] && root=$PARENT
    (cd "$root" && timeout 300 python bench.py --gpus 1 --steps 20 --warmup 3 --no-pipeline --no-t2 \
        --dump-outputs "$OLDPWD/$OUT/dump_$arm") > "$OUT/r04_bench_1gpu_$arm.log" 2>&1
    tail -1 "$OUT/r04_bench_1gpu_$arm.log" | python -c "import json,sys; r=json.loads(sys.stdin.read()); print('$arm', 'ms_per_step', round(r['ms_per_step'], 3), 'ms_dedup', round(r['stages_ms']['ms_dedup'], 3), 'GB/s', round(r['value'], 1), 'parity', r.get('parity_check', {}).get('ok'))"
  done
  python - "$OUT" <<'EOF' | tee "$OUT/r04_bench_dump_compare.txt"
import numpy as np, os, sys
a, b = os.path.join(sys.argv[1], "dump_parent"), os.path.join(sys.argv[1], "dump_new")
for f in sorted(os.listdir(a)):
    x, y = np.load(os.path.join(a, f)), np.load(os.path.join(b, f))
    print(f, x.shape, "identical" if x.shape == y.shape and np.array_equal(x, y) else "DIFFERENT")
EOF
  rm -rf "$OUT/dump_parent" "$OUT/dump_new"
  timeout 270 python bench.py --gpus 1 --steps 10 --warmup 3 > "$OUT/r04_bench_1gpu.log" 2>&1; tail -1 "$OUT/r04_bench_1gpu.log" | cut -c1-400
else
  timeout 540 python tools/fullsize_check.py --config all 2>&1 | tee "$OUT/r04_fullsize_all.jsonl" | cut -c1-300 | tail -20
fi
