#!/bin/bash
# The host program on a config-2 sized sample (180k transcripts, 30 M fragments) written twice from the same
# records: schema 1 (collapsed load, class-plan kernels) and schema 2 with one fp32 weight per hit (per-fragment
# by-length load, segment kernel).  Writes the phase clocks of both runs (MMQ_TIMING, MMQ_LOADER_TIMING) and the
# card's name and power limit to OUT/cli_c2_weighted_timing.txt.
#   tools/gpu_cli_weighted.sh [OUT]      (OUT defaults to profiles)
set -e
OUT=${1:-profiles}
mkdir -p "$OUT"
TMP=$(mktemp -d)
trap 'rm -rf "$TMP"' EXIT
F="$OUT/cli_c2_weighted_timing.txt"
python - "$TMP" <<'PY'
import sys
from mmseq_b200 import synth
s = synth.Synth(20260101 + 2, 180000, 30000000, weights=True)
s.write_hits_fast(sys.argv[1] + "/c2_s1.hits", True)
s.write_hits_fast(sys.argv[1] + "/c2_s2.hits", weights=True)
PY
{
  echo "# mmseq -notraces, default flags, MMQ_TIMING=1 MMQ_LOADER_TIMING=1; $(nproc) host threads"
  nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv
  for s in 1 2; do
    echo
    echo "## schema $s: $(stat -c %s "$TMP/c2_s$s.hits") bytes"
    MMQ_TIMING=1 MMQ_LOADER_TIMING=1 mmseq_b200/bin/mmseq -notraces "$TMP/c2_s$s.hits" "$TMP/out$s" 2>&1 >/dev/null | grep -v "^Counting" || true
  done
  echo
  for ext in .k .M; do cmp -s "$TMP/out1$ext" "$TMP/out2$ext" && echo "$ext byte-identical between schema 1 and 2" || echo "$ext DIFFERS between schema 1 and 2"; done
} > "$F"
cat "$F"
