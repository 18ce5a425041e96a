#!/bin/bash
# Round 3: the 32-byte-record list kernel (B200SPH_PAIR_R32).  One call: the card, build + smoke,
# the GPU suite, the N = 1 dam-break line alternating R32 = 1 / 0 (3 pairs at 20 / 5 steps,
# then 100 / 50 steps each), 8 CTAs / SM for the R32 kernel, and the particle outputs of both
# paths after the timed steps, compared in parity units.
set -u
# output directory: the first argument (default: r03_out)
O=${1:-r03_out}
export O
mkdir -p $O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/r03_gpu.csv 2>&1; cat $O/r03_gpu.csv
timeout 600 python -c "import __graft_entry__ as g; g.build(); g.smoke(); print('smoke ok')" > $O/r03_smoke.log 2>&1
echo "build+smoke rc=$?"; tail -2 $O/r03_smoke.log
timeout 600 python -m pytest tests -m gpu -q > $O/r03_pytest.log 2>&1
echo "pytest rc=$?"; tail -4 $O/r03_pytest.log
B="python bench.py --gpus 1 --no-cpu"
for i in 1 2 3; do
  for r in 1 0; do
    B200SPH_PAIR_R32=$r timeout 300 $B --steps 20 --warmup 5 > $O/r03_alt${i}_r$r.json 2> $O/r03_alt${i}_r$r.err
    echo "alt $i r32=$r rc=$?"
  done
done
for r in 1 0; do
  B200SPH_PAIR_R32=$r timeout 300 $B --steps 100 --warmup 50 --dump-outputs $O/r03_dump_r$r > $O/r03_long_r$r.json 2> $O/r03_long_r$r.err
  echo "long r32=$r rc=$?"
done
B200SPH_PAIR_R32=1 B200SPH_PAIR_MINB=8 timeout 300 $B --steps 20 --warmup 5 --no-extras > $O/r03_minb8_r1.json 2> $O/r03_minb8_r1.err
echo "minb8 rc=$?"
python profiles/r03_compare_dumps.py $O/r03_dump_r1 $O/r03_dump_r0 > $O/r03_dump_compare.json 2>&1; head -c 300 $O/r03_dump_compare.json; echo
rm -rf $O/r03_dump_r1 $O/r03_dump_r0
python - <<'PY'
import json, glob, os
def line(f):
    try:
        d = json.load(open(f))
    except Exception as e:
        return '%s: failed %s' % (f, e)
    r = d['roofline']
    ex = d.get('extra', {})
    tg = ex.get('taylor_green', {}).get('ms_per_step')
    rg = ex.get('rings', {}).get('ms_per_step')
    return '%s ms/step %.4f pair %.4f ms developed %.4f tg %s rings %s' % (
        f.split('/')[-1], d['ms_per_step'], r['avg_launch_ms'], d['developed']['ms_per_step'], tg, rg)
for f in sorted(glob.glob(os.environ['O'] + '/r03_*.json')):
    if 'compare' not in f:
        print(line(f))
PY
