#!/bin/bash
# A/B of CSV registration (tools/bench_csv.py, 30 M records x 6 columns) between a checkout of the parent commit with its
# library built ($1) and this tree, alternated twice in one process tree, then this tree on the dump-style file. One JSON
# line per run in the file $2; the card's name and power limit are in every line.
PARENT=${1:?a checkout of the parent commit with term_b200/libtermgpu.so built}
OUT=${2:?the output file}
HERE=$PWD
mkdir -p "$(dirname "$OUT")"
: > "$OUT"
for rep in 1 2; do
  for tree in "$PARENT" "$HERE"; do
    (cd "$tree" && python tools/bench_csv.py --rows 30000000 --steps 3) | tail -1 | python -c "
import json, sys
d = json.loads(sys.stdin.read()); d['tree'] = '$( [ "$tree" = "$HERE" ] && echo this || echo parent )'; d['rep'] = $rep
print(json.dumps(d))" >> "$OUT"
  done
done
python tools/bench_csv.py --rows 30000000 --steps 3 --dialect dump | tail -1 >> "$OUT"
