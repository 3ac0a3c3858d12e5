#!/bin/bash
# Ceiling of the cfg2 train forward with the row-gather latency taken away, before building anything to hide it.
# Timing-only builds, made from a copy of the working tree with train.cu edited by sed (the tree is not changed):
#   a  the tree as it is
#   b  every head, tail and negative id folded onto 64 rows (`id & 63`) where it is read: the instruction stream is
#      the same, the gathered rows become L1 hits -- and so do the gradient REDs, which now all land on 64 rows
#   c  only the gathers folded (row states and row fragments of head, positive and negative tail read row id & 63);
#      the gradient REDs and touch marks still go to the real rows, so c keeps the scatter of a.  The gathers still
#      wait for the id loads, which stream through L2
#   d  the gathers take no id at all: head, positive and negative rows i & 63, (i + 21) & 63, (i + 42) & 63 of the
#      triple index i.  The ids are still loaded and used by the REDs and touch marks at the end of the iteration, so
#      their latency overlaps the math: what is left is the forward with every load latency of the loop hidden and
#      the scatter of a -- the most a ring that stages rows and ids ahead of the compute warps can reach
# None of b, c and d computes a meaningful model; their losses differ from a's by construction.
#
#   scripts/ring_ceiling_ab.sh build [V..]    build the libraries of variants V (default: a b c d) into build/variants/
#                                             (needs nvcc, no GPU)
#   scripts/ring_ceiling_ab.sh run [PAIRS [V..]]  PAIRS (default 6) rounds of the variants V (default: a b c d), each
#                                             `bench.py --no-extras --no-cpu-baseline --steps 100 --warmup 10`;
#                                             one line per run: build, round, ms_per_step, fwd_ms, adam_ms, final_loss
# Logs go to $RING_CEILING_OUT (default build/ring_ceiling/): the card's name, power limit and max SM clock first.
set -e
cd "$(dirname "$0")/.."
VAR=build/variants
case "$1" in
build)
  shift
  vs=${*:-a b c d}
  for v in $vs; do
    if [ $v = a ]; then bash scripts/build_variant.sh ceil_a >/dev/null; continue; fi
    src=$(mktemp -d)
    cp -r hopwise_b200 include scripts "$src"/
    f=$src/hopwise_b200/csrc/train.cu
    if [ $v = b ]; then
      sed -i \
        -e 's/int64_t h_id = \(is_rec ? __ldg(a\.b\.user + i) : __ldg(a\.b\.head + i)\);/int64_t h_id = (\1) \& 63;/' \
        -e 's/int64_t tp_id = \(is_rec ? __ldg(a\.b\.item + i) : __ldg(a\.b\.tail + i)\);/int64_t tp_id = (\1) \& 63;/' \
        -e 's/int64_t tn_id = __ldg(negs + i);/int64_t tn_id = __ldg(negs + i) \& 63;/' "$f"
    elif [ $v = c ]; then
      sed -i \
        -e 's/row_state(HT, h_id), sr = row_state(RT, r_id), stp = row_state(ET, tp_id);/row_state(HT, h_id \& 63), sr = row_state(RT, r_id), stp = row_state(ET, tp_id \& 63);/' \
        -e 's/int2 stn = row_state(ET, tn_id);/int2 stn = row_state(ET, tn_id \& 63);/' \
        -e 's/frag_load<VEC, G, NCH>(HT\.w\[p\], h_id, /frag_load<VEC, G, NCH>(HT.w[p], h_id \& 63, /' \
        -e 's/frag_load<VEC, G, NCH>(ET\.w\[p\], tp_id, /frag_load<VEC, G, NCH>(ET.w[p], tp_id \& 63, /' \
        -e 's/frag_load<VEC, G, NCH>(ET\.w\[p\], tn_id, /frag_load<VEC, G, NCH>(ET.w[p], tn_id \& 63, /' "$f"
    else
      sed -i \
        -e 's/row_state(HT, h_id), sr = row_state(RT, r_id), stp = row_state(ET, tp_id);/row_state(HT, i \& 63), sr = row_state(RT, r_id), stp = row_state(ET, (i + 21) \& 63);/' \
        -e 's/int2 stn = row_state(ET, tn_id);/int2 stn = row_state(ET, (i + 42) \& 63);/' \
        -e 's/frag_load<VEC, G, NCH>(HT\.w\[p\], h_id, /frag_load<VEC, G, NCH>(HT.w[p], i \& 63, /' \
        -e 's/frag_load<VEC, G, NCH>(ET\.w\[p\], tp_id, /frag_load<VEC, G, NCH>(ET.w[p], (i + 21) \& 63, /' \
        -e 's/frag_load<VEC, G, NCH>(ET\.w\[p\], tn_id, /frag_load<VEC, G, NCH>(ET.w[p], (i + 42) \& 63, /' "$f"
    fi
    n=$(diff hopwise_b200/csrc/train.cu "$f" | grep -c '^>' || true)
    echo "variant $v: $n lines of train.cu edited"
    (cd "$src" && bash scripts/build_variant.sh ceil_$v >/dev/null)
    mkdir -p $VAR && cp "$src/$VAR/libkge_b200_ceil_$v.so" $VAR/
    rm -rf "$src"
  done
  for v in $vs; do ls -l $VAR/libkge_b200_ceil_$v.so; done
  ;;
run)
  pairs=${2:-6}
  shift; shift || true
  vs=${*:-a b c d}
  out=${RING_CEILING_OUT:-build/ring_ceiling}
  mkdir -p $out
  nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $out/card.txt
  for i in $(seq 1 "$pairs"); do
    for v in $vs; do
      KGE_B200_LIB=$PWD/$VAR/libkge_b200_ceil_$v.so python bench.py --gpus 1 --steps 100 --warmup 10 --no-extras \
        --no-cpu-baseline 2>>$out/stderr.txt | python -c "
import json, sys
d = json.loads(sys.stdin.readline())
r = d['roofline']
print('$v', $i, round(d['ms_per_step'], 5), round(r['fwd_ms'], 5), round(r['adam_ms'], 5), d['final_loss'])" | tee -a $out/ab.log
    done
  done
  ;;
*)
  echo "usage: $0 build | run [PAIRS]" >&2
  exit 2
  ;;
esac
