#!/bin/bash
# Pruned tail (T11 / V5 on the pooled rows only) A/B on one B200, in one call.  A = VB200_PRUNE=0 (full tail), B = VB200_PRUNE=1
# (default).  Usage: scripts/r3_pruned_tail.sh OUT_DIR (relative to the repository root).  Writes the raw lines under OUT_DIR and
# a summary (scripts/r3_pruned_tail_summary.py) to OUT_DIR/summary.md.
#   1. card name, power limit, max SM clock
#   2. outputs of both arms, dumped and compared with np.array_equal (VQA with the per-launch table, multitask)
#   3. ABBA x 4 pairs: 200 steps (under the power cap) and 40 steps (burst)
#   4. reported, not gated: batch 512, retrieval 250 x 250 (multitask comes from step 2)
O=${1:?usage: scripts/r3_pruned_tail.sh OUT_DIR}
cd "$(dirname "$0")/.."
mkdir -p $O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/env.txt
run() {   # run <arm> <tag> <bench args...>
    local arm=$1 tag=$2; shift 2
    VB200_PRUNE=$arm timeout 600 python bench.py --no-cpu-baseline "$@" > $O/$tag.json 2> $O/$tag.err
    echo "$tag exit $?"
}
for a in 0 1; do
    run $a dump_vqa_p$a --steps 40 --dump-outputs $O/dump_vqa_p$a --ops-table $O/ops_p$a.jsonl
    run $a dump_mt_p$a --steps 40 --workload multitask --dump-outputs $O/dump_mt_p$a
done
for i in 1 2 3 4; do
    if [ $((i % 2)) -eq 1 ]; then order="0 1"; else order="1 0"; fi          # A B, B A, A B, B A
    for a in $order; do run $a s200_p${a}_$i; done
    for a in $order; do run $a s40_p${a}_$i --steps 40; done
done
for a in 0 1; do
    run $a b512_p$a --steps 40 --batch 512
    run $a retr_p$a --workload retrieval --captions 250 --images 250 --steps 1
done
python scripts/r3_pruned_tail_summary.py $O > $O/summary.md 2>&1
cat $O/summary.md
