#!/bin/sh
# tools/reloc_staged_sharded.py at 1, 2, 4 and 8 GPUs, one JSON line each, into $1 (default
# profiles/r7_reloc_staged_sharded.jsonl, replaced).  Run from the repository root on a box with 8 GPUs.
set -e
out=${1:-profiles/r7_reloc_staged_sharded.jsonl}
rm -f "$out"
python tools/reloc_staged_sharded.py --out "$out"
for n in 2 4 8; do
    python -m torch.distributed.run --standalone --nproc-per-node "$n" tools/reloc_staged_sharded.py --out "$out"
done
