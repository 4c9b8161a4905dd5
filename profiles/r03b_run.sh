#!/bin/bash
# round 3, call b: whole GPU suite and smoke on the per-atom branch; bench.py of the parent commit and of this branch
# alternated on the same box, with --dump-outputs of each run compared.  _parent/ (not part of the repository) is a
# checkout of the parent commit built with `python -m distmlip_b200.build` before the call.
cd "$(dirname "$0")/.."
O=${1:?usage: $0 OUTPUT_DIR}
mkdir -p $O
timeout 1500 python -m pytest tests -m gpu -q -rs > $O/r03b_pytest.txt 2>&1
tail -4 $O/r03b_pytest.txt
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $O/r03b_smoke.txt 2>&1
echo "smoke rc $?"; tail -2 $O/r03b_smoke.txt
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/r03b_bench_ab.txt
for i in 1 2; do
  for arm in parent branch; do
    dir=.; [ $arm = parent ] && dir=_parent
    (cd $dir && timeout 400 python bench.py --gpus 1 --steps 10 --warmup 3 --no-cpu-baseline \
       --dump-outputs /tmp/dump_1M_${arm}_$i > /tmp/b_1M_${arm}_$i.json 2>/dev/null)
    (cd $dir && timeout 300 python bench.py --gpus 1 --steps 10 --warmup 3 --model tensornet --cells 23 \
       --dump-outputs /tmp/dump_tn_${arm}_$i > /tmp/b_tn_${arm}_$i.json 2>/dev/null)
  done
done
python - >> $O/r03b_bench_ab.txt <<'PY'
import glob, json, os
import numpy as np
def line(p):
    try:
        return json.loads([l for l in open(p) if l.startswith('{')][-1])
    except Exception as ex:
        return {"error": str(ex)}
for w in ("1M", "tn"):
    for i in (1, 2):
        for arm in ("parent", "branch"):
            d = line(f"/tmp/b_{w}_{arm}_{i}.json")
            print(w, arm, i, "value", d.get("value"), "ms_per_step", d.get("ms_per_step"), d.get("error", ""))
    def dump(arm, i):
        return {os.path.basename(f): np.load(f) for f in sorted(glob.glob(f"/tmp/dump_{w}_{arm}_{i}/*.npy"))}
    p1, p2, b1, b2 = dump("parent", 1), dump("parent", 2), dump("branch", 1), dump("branch", 2)
    for k in p1:
        dd = lambda a, b: float(np.abs(a[k].astype(np.float64) - b[k].astype(np.float64)).max()) if k in b else None
        print(f"{w} {k}: max|parent1-parent2| {dd(p1, p2)}  max|parent1-branch1| {dd(p1, b1)}  "
              f"max|parent2-branch2| {dd(p2, b2)}  max|branch1-branch2| {dd(b1, b2)}  max|x| {float(np.abs(p1[k]).max())}")
PY
cat $O/r03b_bench_ab.txt
