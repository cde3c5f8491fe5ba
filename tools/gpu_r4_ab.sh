#!/bin/bash
# A/B of the emulation kernel on one GPU: the parent commit's library (pokegym_b200/csrc/variants/libgbenv_parent.so, built
# from the parent's sources with build()'s flags) against the in-tree build.
#   tools/gpu_r4_ab.sh verify OUTDIR   build, pipe map, smoke(), the GPU tests, byte comparison of bench.py --dump-outputs
#   tools/gpu_r4_ab.sh bench OUTDIR    the pipe map, then parent and new alternately, three full bench.py runs each
#   tools/gpu_r4_ab.sh pipes OUTDIR    the pipe map only
# Records go to OUTDIR: card.txt, pipes_b200.json, pytest_gpu.log, dump_compare.txt, r4_bench_parent.jsonl, r4_bench.jsonl.
cd "$(dirname "$0")/.."
MODE=$1; OUT=${2:?usage: tools/gpu_r4_ab.sh verify|bench|pipes OUTDIR}
mkdir -p "$OUT"
PARENT=$PWD/pokegym_b200/csrc/variants/libgbenv_parent.so
python -c "import __graft_entry__ as g; g.build()" || exit 1
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee -a "$OUT/card.txt"
python tools/bench_pipes.py --out "$OUT/pipes_b200.json" > /dev/null && echo pipes ok
[ "$MODE" = pipes ] && exit 0
if [ "$MODE" = verify ]; then
  python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
  timeout 900 python -m pytest -q -m gpu tests/ > "$OUT/pytest_gpu.log" 2>&1; tail -2 "$OUT/pytest_gpu.log"
  D=$(mktemp -d)
  GBENV_LIB=$PARENT python bench.py --gpus 1 --steps 200 --warmup 20 --legs none --dump-outputs $D/parent > /dev/null 2>&1
  python bench.py --gpus 1 --steps 200 --warmup 20 --legs none --dump-outputs $D/new > /dev/null 2>&1
  for f in $D/parent/*; do cmp -s $f $D/new/$(basename $f) && echo "identical $(basename $f)" || echo "DIFFERS $(basename $f)"; done | tee "$OUT/dump_compare.txt"
  rm -rf $D
  exit 0
fi
for i in 1 2 3; do
  date +%T
  GBENV_LIB=$PARENT python bench.py --gpus 1 --steps 200 --warmup 20 2>/dev/null | grep '^{' >> "$OUT/r4_bench_parent.jsonl"
  python bench.py --gpus 1 --steps 200 --warmup 20 2>/dev/null | grep '^{' >> "$OUT/r4_bench.jsonl"
  nvidia-smi --query-gpu=name,power.limit --format=csv,noheader >> "$OUT/card.txt"
done
OUT="$OUT" python - <<'PY'
import json, os
for n in ("r4_bench_parent", "r4_bench"):
    for l in open(os.path.join(os.environ["OUT"], f"{n}.jsonl")):
        d = json.loads(l)
        lb = d.get("large_batch")
        print(n, round(d["value"]), {k: round(v["value"], 1) for k, v in d["legs"].items() if isinstance(v, dict) and "value" in v},
              round(lb["value"]) if isinstance(lb, dict) and "value" in lb else lb)
PY
