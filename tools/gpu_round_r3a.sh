#!/bin/bash
# Round r3a: P resident in tensor memory.  Parity of the new decoder path, then the A/B of the parent build
# (tools/ab/parent: a built checkout of the parent commit) against the in-tree build, alternating on one box.
# Usage: tools/gpu_round_r3a.sh OUTDIR   (bench JSON lines and test summaries are written there)
OUT=${1:?usage: tools/gpu_round_r3a.sh OUTDIR}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/card.txt

echo "=== parity: TMEM vs L2 path, bitwise"
timeout 900 python -m pytest -q -m gpu tests/test_gpu_dec_tmem.py -s 2>&1 | tail -15 | tee $OUT/pytest_tmem.txt

row() {   # label, tree, extra args
  (cd $2 && timeout 300 python bench.py --steps 20 --warmup 3 --no-cpu-baseline --no-train ${@:3} 2>/dev/null | tail -1) > $OUT/bench_$1.json
  python -c "import json; d=json.load(open('$OUT/bench_$1.json')); print('$1', round(d['value']), d['ms_per_step'], round(d['roofline']['decoder_step_us'],2), d['kernel_ms_per_step']['dec_scan'])"
}
echo "=== A/B (label value ms_per_step decoder_step_us dec_scan_ms)"
P=$PWD/tools/ab/parent
row old1 $P --dump-outputs /tmp/dump_old
row new1 $PWD --dump-outputs /tmp/dump_new
row old2 $P
row new2 $PWD
row old3 $P
row new3 $PWD
python - <<'EOF'
import os, hashlib
for f in sorted(os.listdir('/tmp/dump_old')):
    a = open('/tmp/dump_old/' + f, 'rb').read(); b = open('/tmp/dump_new/' + f, 'rb').read()
    print('dump', f, len(a), 'identical' if a == b else 'DIFFERENT', hashlib.sha256(a).hexdigest()[:16])
EOF

echo "=== phase traces"
for arm in old new; do
  T=$PWD; [ $arm = old ] && T=$P
  echo "--- $arm"
  (cd $T && LVSR_DEC_TRACE=1 timeout 300 python bench.py --steps 1 --warmup 1 --no-cpu-baseline --no-train 2>&1 | grep "dec_scan trace\] \(CTA\|attention row\)" | tail -3)
done
echo "--- new, LVSR_DEC_TMEM_P=0"
LVSR_DEC_TMEM_P=0 LVSR_DEC_TRACE=1 timeout 300 python bench.py --steps 1 --warmup 1 --no-cpu-baseline --no-train 2>&1 | grep "dec_scan trace\] \(CTA\|attention row\)" | tail -3

echo "=== full GPU suite + smoke"
timeout 1500 python -m pytest -q -m gpu tests 2>&1 | tail -15 | tee $OUT/pytest_gpu.txt
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2

echo "=== workspace placement sweep"
for kb in 0 2048 4096 6144; do
  for arm in old new; do
    T=$PWD; [ $arm = old ] && T=$P
    (cd $T && LVSR_WS_SHIFT_KB=$kb timeout 300 python bench.py --steps 20 --warmup 3 --no-cpu-baseline --no-train 2>/dev/null | tail -1) > $OUT/ws_${arm}_$kb.json
    python -c "import json; d=json.load(open('$OUT/ws_${arm}_$kb.json')); print('shift $kb $arm', round(d['value']), d['ms_per_step'], round(d['roofline']['decoder_step_us'],2))"
  done
done
