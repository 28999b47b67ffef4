#!/bin/bash
# A/B of two strict-fp libraries on one B200, in one run: card, power limit and clocks, the whole GPU suite and the smoke run
# on this tree's library, then a baseline library (BASE) and this tree's alternated three times with scripts/quick_bench.py
# (xpbd_step kernel us, L2-warm) and bench.py (frame, roofline.kernel_ms), and the --dump-outputs of both compared byte for byte.
# Usage: bash scripts/xpbd_lib_ab.sh BASE_LIB [OUT_DIR]   (BASE_LIB: e.g. build_variant() output of the parent commit's sources)
cd "$(dirname "$0")/.."
BASE=$1
O=${2:-$(mktemp -d)}; echo "outputs in $O"
NEW=newton_b200/libnewton_b200.so
mkdir -p "$O"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm,clocks.mem --format=csv
timeout -k 5 1200 python -m pytest -q -m gpu tests 2>&1 | tail -4
timeout -k 5 300 python scripts/smoke_entry.py 2>&1 | tail -1
for i in 1 2 3; do
  for lib in "$BASE" "$NEW"; do
    echo "=== quick_bench $i $lib"; NB2_LIB=$lib timeout -k 5 200 python scripts/quick_bench.py 4096 8 quad xpbd 2>&1 | tail -2
  done
done
for i in 1 2 3; do
  for lib in "$BASE" "$NEW"; do
    echo "=== bench $i $lib"
    NB2_LIB=$lib timeout -k 5 300 python bench.py --gpus 1 --steps 200 --warmup 10 --no-cpu-baseline --no-fast-twin 2>/dev/null |
      python -c "import json,sys; r=json.loads([l for l in sys.stdin if l.startswith('{')][-1]); print(r['value'], r['ms_per_step'], r['roofline']['kernel_ms'], r.get('clocks'))"
  done
done
for tag in base new; do
  lib=$BASE; [ $tag = new ] && lib=$NEW
  NB2_LIB=$lib timeout -k 5 300 python bench.py --gpus 1 --steps 20 --warmup 5 --no-cpu-baseline --no-fast-twin --dump-outputs "$O/dump_$tag" > /dev/null 2>&1
done
python - "$O" <<'PY'
import os, sys, numpy as np
o = sys.argv[1]
names = sorted(os.listdir(os.path.join(o, "dump_base")))
same = [n for n in names if open(os.path.join(o, "dump_base", n), "rb").read() == open(os.path.join(o, "dump_new", n), "rb").read()]
print(f"--dump-outputs: {len(same)}/{len(names)} files byte-identical", sorted(set(names) - set(same)))
PY
