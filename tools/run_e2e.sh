#!/usr/bin/env bash
# End-to-end drop-in check on a GPU box: the reference's OWN annealing driver and moves (gaml.cc, moves.cc,
# compiled unchanged) once over the reference ProbCalculator (gaml_ref) and once over the CUDA one (gaml_gpu),
# same synthetic LastGraph + FASTQ input, same seeds. Traces must be identical; wall times give SA it/s.
set -uo pipefail
ROOT="$(cd "$(dirname "$0")/.." && pwd)"
OUT=${1:-$ROOT/gpurun_out/e2e}
ITERS=${2:-500}
KINDS=${E2E_KINDS:-"single paired"}     # E2E_KINDS=paired E2E_UNIQUE=100 E2E_READS=400000: a 1 Mbp / 400 k-pair run
UNIQUE=${E2E_UNIQUE:-10}
READS=${E2E_READS:-50000}
PENALTY=()                               # E2E_PENALTY="<penalty_constant> <penalty_step>": the paired set's coverage-gap penalty
if [ -n "${E2E_PENALTY:-}" ]; then
  read -r pc ps <<< "$E2E_PENALTY"
  PENALTY=(--penalty-constant "$pc" --penalty-step "$ps")
fi
mkdir -p "$OUT"
rc=0
for kind in $KINDS; do
  D=/tmp/e2e_$kind
  rm -rf "$D"
  python "$ROOT/tools/make_e2e_dataset.py" "$D" --kind $kind --n-unique "$UNIQUE" --n-reads "$READS" --iterations "$ITERS" "${PENALTY[@]}" > "$OUT/$kind.gen.log"
  t0=$(date +%s.%N)
  ( cd "$D" && stdbuf -oL "$ROOT/oracle/_ref/gaml_ref" gaml.cfg > ref.log 2>&1 )
  t1=$(date +%s.%N)
  ( cd "$D" && stdbuf -oL "$ROOT/oracle/_ref/gaml_gpu" gaml.cfg > gpu.log 2>&1 ) || { echo "gaml_gpu failed ($kind)"; tail -5 "$D/gpu.log"; rc=1; }
  t2=$(date +%s.%N)
  python -c "print('%.2f' % ($t1 - $t0))" > "$D/ref.time"; python -c "print('%.2f' % ($t2 - $t1))" > "$D/gpu.time"
  python "$ROOT/tools/compare_traces.py" "$D/ref.log" "$D/gpu.log" | tee "$OUT/$kind.compare.txt" || rc=1
  echo "$kind: reference $(cat $D/ref.time)s, cuda $(cat $D/gpu.time)s for $ITERS iterations (wall, includes read loading and the one-off CPU alignment of new keys)" | tee -a "$OUT/$kind.compare.txt"
  # the annealing loop alone: wall time between the first and the last trace line (gaml.cc:330 prints hh:mm:ss) is too coarse,
  # so the loop is timed by the "start prob" line's position: seconds from that line to the end of the log
  python - "$D/ref.log" "$D/gpu.log" <<'PY' | tee -a "$OUT/$kind.compare.txt"
import sys
for p in sys.argv[1:]:
    n = sum(1 for l in open(p, errors="replace") if l.startswith("itnum "))
    print(f"{p}: {n} annealing iterations")
PY
  if [ -x "$ROOT/oracle/_ref/gaml_gpu_batched" ]; then
    # the same driver with the moves' candidate lists scored in device batches (oracle/build_ref.sh, gaml_gpu_batched)
    t3=$(date +%s.%N)
    ( cd "$D" && stdbuf -oL "$ROOT/oracle/_ref/gaml_gpu_batched" gaml.cfg > batched.log 2>&1 ) || { echo "gaml_gpu_batched failed ($kind)"; tail -5 "$D/batched.log"; rc=1; }
    t4=$(date +%s.%N)
    python "$ROOT/tools/compare_traces.py" "$D/ref.log" "$D/batched.log" | tee "$OUT/$kind.batched.compare.txt" || rc=1
    python -c "print('$kind: cuda with batched moves %.2f s for $ITERS iterations' % ($t4 - $t3))" | tee -a "$OUT/$kind.batched.compare.txt"
    cp "$D/batched.log" "$OUT/$kind.batched.log"
  fi
  grep -c "^itnum" "$D/gpu.log" > /dev/null
  cp "$D/ref.log" "$OUT/$kind.ref.log"; cp "$D/gpu.log" "$OUT/$kind.gpu.log"
done
exit $rc
