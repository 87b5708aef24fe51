#!/bin/bash
# compute-sanitizer evidence for one learner step of every kernel family (SURVEY.md §5; VERDICT r1 item 9).
# Run on a GPU machine:  bash tools/sanitize.sh   -> $OUT/sanitizer_*.log, OUT defaults to sanitizer_logs/ (copy the summaries to profiles/)
# racecheck covers shared-memory hazards inside a block; the tcgen05 / TMA (async proxy) traffic is invisible to it, so
# the mbarrier pipelines are additionally covered by the parity tests (stale shared-memory poisoning, 30-run bias-sum stress).
set -u
cd "$(dirname "$0")/.."
OUT=${OUT:-sanitizer_logs}
mkdir -p "$OUT"
CS=${CS:-/usr/local/cuda/bin/compute-sanitizer}
for tool in memcheck racecheck synccheck initcheck; do
  echo "== $tool" | tee "$OUT/sanitizer_$tool.log"
  timeout 900 $CS --tool $tool --print-limit 20 python tests/diag/sanitize_step.py ${MODES:-bf16 split three lstm ops} >> "$OUT/sanitizer_$tool.log" 2>&1
  echo "exit code $?" >> "$OUT/sanitizer_$tool.log"
  grep -E "ERROR SUMMARY|RACECHECK SUMMARY|exit code|total_loss|ops: ok" "$OUT/sanitizer_$tool.log" | tail -14
done
