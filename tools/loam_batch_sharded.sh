#!/bin/sh
# tools/loam_batch_sharded.py at 1, 2, 4 and 8 GPUs, one JSON line each, into $1 (default
# profiles/r9_loam_batch_sharded.jsonl, replaced).  Run from the repository root.  A width the box has too few GPUs for
# is not measured: it runs with every rank on GPU 0 instead (--share-gpu0, one repetition), a results check whose line
# goes to the same name with _shared_gpu0 (replaced) and whose times are not scaling numbers.
set -e
out=${1:-profiles/r9_loam_batch_sharded.jsonl}
shared=${out%.jsonl}_shared_gpu0.jsonl
gpus=$(nvidia-smi -L | wc -l)
rm -f "$out" "$shared"
python tools/loam_batch_sharded.py --out "$out"
for n in 2 4 8; do
    if [ "$n" -le "$gpus" ]; then
        python -m torch.distributed.run --standalone --nproc-per-node "$n" tools/loam_batch_sharded.py --out "$out"
    else
        echo "$n GPUs: not measured ($gpus visible); results check with $n ranks on GPU 0"
        python -m torch.distributed.run --standalone --nproc-per-node "$n" tools/loam_batch_sharded.py --share-gpu0 \
            --reps 1 --warmup 0 --out "$shared"
    fi
done
