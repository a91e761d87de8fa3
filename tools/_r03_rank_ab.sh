#!/bin/bash
# Round 3 measurements of the small-tie-group ranking (profiles/r03_*), written to OUTDIR:
#   tools/_r03_rank_ab.sh OUTDIR check   the new tests, smoke(), the A/B of tools/rank_ab.py with a
#                                        per-kernel profile
#   tools/_r03_rank_ab.sh OUTDIR bench   bench.py with and without PFPB200_RANK_WARP_PASSES=1 (outputs
#                                        dumped and compared)
#   tools/_r03_rank_ab.sh OUTDIR suite   the whole GPU suite
set -u
OUT=${1:?usage: _r03_rank_ab.sh OUTDIR check|bench|suite}
WHAT=${2:?usage: _r03_rank_ab.sh OUTDIR check|bench|suite}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/r03_card.txt"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/r03_build.log" 2>&1 || { tail -30 "$OUT/r03_build.log"; exit 1; }
if [ "$WHAT" = check ]; then
  timeout 900 python -m pytest -q tests/test_rank_small_groups_gpu.py 2>&1 | tee "$OUT/r03_pytest_small_groups.log" | tail -15
  timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tee "$OUT/r03_smoke.log" | tail -3
  timeout 900 python tools/rank_ab.py --profile "$OUT" 2>&1 | tee "$OUT/r03_rank_ab.log"
elif [ "$WHAT" = bench ]; then
  for arm in 0 1; do
    PFPB200_RANK_WARP_PASSES=$arm timeout 270 python bench.py --gpus 1 --steps 20 --warmup 3 --no-pipeline --no-t2 \
        --dump-outputs "$OUT/dump_warp_passes_$arm" > "$OUT/r03_bench_warp_passes_$arm.log" 2>&1
    tail -1 "$OUT/r03_bench_warp_passes_$arm.log" | python -c "import json,sys; r=json.loads(sys.stdin.read()); print('PFPB200_RANK_WARP_PASSES=$arm', 'ms_per_step', round(r['ms_per_step'], 3), 'ms_rank', round(r['stages_ms']['ms_rank'], 3), 'GB/s', round(r['value'], 1), 'parity ok', r.get('parity_check', {}).get('ok'))"
  done
  python - "$OUT" <<'EOF' | tee "$OUT/r03_dump_compare.txt"
import numpy as np, os, sys
a, b = os.path.join(sys.argv[1], "dump_warp_passes_0"), os.path.join(sys.argv[1], "dump_warp_passes_1")
for f in sorted(os.listdir(a)):
    x, y = np.load(os.path.join(a, f)), np.load(os.path.join(b, f))
    print(f, x.shape, "identical" if x.shape == y.shape and np.array_equal(x, y) else "DIFFERENT")
EOF
  rm -rf "$OUT/dump_warp_passes_0" "$OUT/dump_warp_passes_1"
else
  timeout 540 python -m pytest -q -m gpu tests 2>&1 | tee "$OUT/r03_pytest_gpu.log" | tail -15
fi
