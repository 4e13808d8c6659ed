#!/bin/bash
# RAD-TEAM epoch records on one GPU box: build + smoke, the GPU suite, tools/radteam_epoch.py, and bench.py's maps leg and
# headline run alternately on a checkout of an earlier commit (its own Python and library) and on this tree.
#   bash tools/gpu_radteam.sh <output directory> <directory of the earlier checkout, built> [reps]
out=$1; old=$2; reps=${3:-3}
mkdir -p $out
python -c "import __graft_entry__ as g; g.build(); g.smoke()" 2>&1 | tail -2
timeout 1500 python -m pytest tests -m gpu -q -p no:cacheprovider > $out/pytest_gpu.log 2>&1; echo "pytest rc=$?"
tail -3 $out/pytest_gpu.log
timeout 900 python tools/radteam_epoch.py --out $out/radteam 2>&1 | tail -3; echo "radteam_epoch rc=$?"
b="python bench.py --gpus 1 --steps 240 --warmup 24 --legs maps --no-cpu-baseline"
for i in $(seq 1 $reps); do
  echo "== old $i"; (cd $old && timeout 400 $b 2>&1 | tail -1) > $out/bench_old_$i.json
  echo "== new $i"; timeout 400 $b 2>&1 | tail -1 > $out/bench_new_$i.json
done
OUT=$out python - <<'PY'
import glob, json, os
for f in sorted(glob.glob(os.path.join(os.environ["OUT"], "bench_*.json"))):
    try:
        d = json.load(open(f)); print(f, "value %.4g" % d["value"], "maps.update_ms %.5f" % d["maps"]["update_ms"])
    except Exception as e:
        print(f, "unreadable:", open(f).read()[-400:])
PY
