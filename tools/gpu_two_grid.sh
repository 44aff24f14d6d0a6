# tools/gpu_two_grid.sh [-r rounds] [-t tag] [-o dir] [-a "bench args"] V1 V2 ...: bench.py's default workload on libbbenv_<V>.so variants
# (csrc/Makefile `variant`, e.g. V=t84 VFLAGS="-DBB_TWO_WARPS=8 -DBB_TWO_MIN_BLOCKS=4"; the name `stock` is libbbenv.so), alternated
# within one process tree: every round runs each library once, the order reversed on every other round, so that a drift of
# the card (clocks, neighbours) falls on all of them alike.  One line per run (M env-steps/s, k_run ms, with_gb, parity),
# then min / median / max per library.  The card's name, power limit and SM clocks are read at the start and at the end.
# Each run's JSON line and stderr go to <dir> (default: a new temporary directory).
cd "$(dirname "$0")/.."
rounds=3; extra=""; tag=grid; dir=""
while [ $# -gt 0 ]; do case $1 in -r) rounds=$2; shift 2;; -a) extra="$2"; shift 2;; -t) tag=$2; shift 2;; -o) dir=$2; shift 2;; *) break;; esac; done
libs="$*"
[ -n "$dir" ] || dir=$(mktemp -d); mkdir -p "$dir"; echo "results: $dir"
rev=$(echo $libs | tr ' ' '\n' | tac | tr '\n' ' ')
smi() { nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm --format=csv,noheader; }
echo "gpu: $(smi)"
for r in $(seq 1 $rounds); do
  order=$libs; [ $((r % 2)) -eq 0 ] && order=$rev
  for v in $order; do
    if [ $v = stock ]; then unset BBENV_LIB; else export BBENV_LIB=$PWD/deepgroebner_b200/libbbenv_$v.so; fi
    out=$dir/${tag}_${v}_$r
    timeout 300 python bench.py --gpus 1 --steps 20 --warmup 3 --no-cpu --no-extras $extra > $out.json 2> $out.err
    python -c "
import json
d = json.loads(open('$out.json').read())
k = {n: round(t, 4) for n, t in d['kernel_ms'].items() if n != 'how'}
print('$v', $r, round(d['value'] / 1e6, 1), 'M', 'kernel_ms', k, 'with_gb', round(d['with_gb']['value'] / 1e6, 1), 'M',
      'parity', d['parity']['episodes_checked'], d['parity']['mismatches'], 'slots', d['config']['slots'], 'clocks', d.get('clocks'))
" 2>/dev/null || { echo "$v $r FAILED"; tail -3 $out.err; }
  done
done
python - "$dir" $tag $libs <<'EOF'
import glob, json, sys
import numpy as np
for v in sys.argv[3:]:
    x = [json.loads(open(f).read())['value'] / 1e6 for f in sorted(glob.glob('%s/%s_%s_*.json' % (sys.argv[1], sys.argv[2], v))) if open(f).read().strip()]
    if x:
        print('%-8s n=%d  min %.1f  median %.1f  max %.1f  M env-steps/s' % (v, len(x), min(x), float(np.median(x)), max(x)))
EOF
echo "gpu: $(smi)"
