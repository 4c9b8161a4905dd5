#!/bin/bash
# round 3, call a: per-atom energies / virials -- the new GPU tests (observed errors printed), the backward-phase cost
# of the per-atom path (tests/peratom_time.py), one compute-sanitizer memcheck of the per-atom path
cd "$(dirname "$0")/.."
O=${1:?usage: $0 OUTPUT_DIR}
mkdir -p $O
timeout 900 python -m pytest tests/test_gpu_peratom.py -m gpu -q -s -rs > $O/r03a_pytest_peratom.txt 2>&1
tail -3 $O/r03a_pytest_peratom.txt
timeout 600 python tests/peratom_time.py 12 > $O/r03a_peratom_time.txt 2>&1
cat $O/r03a_peratom_time.txt
timeout 600 compute-sanitizer --tool memcheck --leak-check no python - > $O/r03a_memcheck_peratom.txt 2>&1 <<'PY'
import numpy as np
from distmlip_b200.structures import si_diamond
from tests._util import engine_from_model, make_model
from tests.test_gpu_tensornet import tn_engine
from tests.test_oracle_tensornet import make_tn
atoms = si_diamond(2, nz=8, seed=1)
sp = np.zeros(len(atoms), dtype=np.int32)
for label, eng in (("chgnet 1 partition", engine_from_model(make_model())),
                   ("chgnet 2-partition group", engine_from_model(make_model(), device=[0, 0])),
                   ("tensornet 1 partition", tn_engine(make_tn(seed=3, scale=1.5))),
                   ("tensornet 2-partition group", tn_engine(make_tn(seed=3, scale=1.5), device=[0, 0]))):
    eng.set_structure(atoms.get_positions(), atoms.get_cell(), sp, np.ones(3, dtype=np.int32))
    e, f, s, ae, aw = eng.compute_peratom()
    print(label, "E", e, "sum e_i", ae.sum(), "max|W|", np.abs(aw).max(), flush=True)
    eng.close()
PY
tail -4 $O/r03a_memcheck_peratom.txt
