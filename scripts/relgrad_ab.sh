#!/bin/bash
# A/B of the train step between two builds of the library, alternating bench.py runs on one GPU.
#
#   scripts/relgrad_ab.sh build [REV]     build REV (default: main) and the working tree into build/variants/
#                                         as libkge_b200_main.so and libkge_b200_branch.so (needs git and nvcc, no GPU)
#   scripts/relgrad_ab.sh run [PAIRS]     PAIRS (default 6) alternating runs of
#                                         `bench.py --no-extras --no-cpu-baseline --steps 100 --warmup 10`, main first;
#                                         one line per run: build, pair, ms_per_step, fwd_ms, adam_ms, final_loss.
#                                         Then one --dump-outputs run per build and the largest table difference.
# Logs go to $RELGRAD_AB_OUT (default build/relgrad_ab/): the card's name, power limit and clocks first.
set -e
cd "$(dirname "$0")/.."
VAR=build/variants
case "$1" in
build)
  rev=${2:-main}
  src=$(mktemp -d)
  git archive "$rev" | tar -x -C "$src"
  (cd "$src" && bash scripts/build_variant.sh main >/dev/null)
  mkdir -p $VAR && cp "$src/$VAR/libkge_b200_main.so" $VAR/
  rm -rf "$src"
  bash scripts/build_variant.sh branch >/dev/null
  ls -l $VAR/libkge_b200_main.so $VAR/libkge_b200_branch.so
  ;;
run)
  pairs=${2:-6}
  out=${RELGRAD_AB_OUT:-build/relgrad_ab}
  mkdir -p $out
  nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $out/card.txt
  for i in $(seq 1 "$pairs"); do
    for v in main branch; do
      KGE_B200_LIB=$PWD/$VAR/libkge_b200_$v.so python bench.py --gpus 1 --steps 100 --warmup 10 --no-extras \
        --no-cpu-baseline 2>>$out/stderr.txt | python -c "
import json, sys
d = json.loads(sys.stdin.readline())
r = d['roofline']
print('$v', $i, round(d['ms_per_step'], 5), round(r['fwd_ms'], 5), round(r['adam_ms'], 5), d['final_loss'])" | tee -a $out/ab.log
    done
  done
  tmp=$(mktemp -d)
  for v in main branch; do
    KGE_B200_LIB=$PWD/$VAR/libkge_b200_$v.so python bench.py --gpus 1 --no-extras --no-cpu-baseline \
      --dump-outputs $tmp/$v 2>>$out/stderr.txt >/dev/null
  done
  python - "$tmp" <<'EOF' | tee $out/dump_compare.txt
import os, sys
import numpy as np
sys.path.insert(0, "tests")
from kge_helpers import assert_weights_close
d = sys.argv[1]
for f in sorted(os.listdir(os.path.join(d, "main"))):
    a, b = np.load(os.path.join(d, "main", f)), np.load(os.path.join(d, "branch", f))
    print(f, a.shape, "max abs diff", float(np.abs(a - b).max()))
    if f == "loss.npy":
        np.testing.assert_allclose(b, a, rtol=1e-5)
    else:
        assert_weights_close(b, a, outlier_atol=5e-3, err_msg=f)
print("dumped outputs agree")
EOF
  rm -rf "$tmp"
  ;;
*)
  echo "usage: $0 build [REV] | run [PAIRS]" >&2
  exit 2
  ;;
esac
