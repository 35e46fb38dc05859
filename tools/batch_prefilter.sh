#!/bin/sh
# tools/batch_prefilter.py: the batch measurement (S = 512 and 4096), then the single-cloud regression check with the
# parent commit's package and this one alternating, three runs each, one JSON line per run into $1 (default
# profiles/r11_batch_prefilter.jsonl, replaced).  $2: a checkout of the parent commit whose libraries are built (make -C
# loc_lib_b200/csrc there); without it the regression check is skipped.  Run from the repository root after build().
set -e
out=${1:-profiles/r11_batch_prefilter.jsonl}
rm -f "$out"
python tools/batch_prefilter.py --mode batch --out "$out"
if [ -n "$2" ]; then
    for i in 1 2 3; do
        python tools/batch_prefilter.py --mode single --tag parent --root "$2" --out "$out"
        python tools/batch_prefilter.py --mode single --tag this --out "$out"
    done
fi
