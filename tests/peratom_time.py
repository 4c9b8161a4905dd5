"""Diagnostic (not a test): device time of the backward phase (b2m_last_timings[2]: the edge-final kernels, the per-atom
energy kernel and any all-reduce included) with and without per-atom output, on the resident graph.  The two modes run
in alternating order after warm-up; the wall time of a whole call (host copies included) is printed beside it.
    usage: python tests/peratom_time.py [reps]"""
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from distmlip_b200.implementations.matgl import CHGNet_Dist, Potential_Dist, TensorNet_Dist  # noqa: E402
from distmlip_b200.random_init import RandomCHGNet, RandomTensorNet  # noqa: E402
from distmlip_b200.structures import si_diamond  # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 12
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                     capture_output=True, text=True).stdout.strip(), flush=True)
for label, make, cells in (("chgnet", lambda: CHGNet_Dist.from_existing(RandomCHGNet(seed=0)), 23),
                           ("chgnet", lambda: CHGNet_Dist.from_existing(RandomCHGNet(seed=0)), 50),
                           ("tensornet", lambda: TensorNet_Dist.from_existing(RandomTensorNet(seed=0)), 23)):
    model = make()
    model.enable_distributed_mode([0])
    pot = Potential_Dist(model=model, calc_forces=True, calc_stresses=True)
    atoms = si_diamond(cells)
    pot(atoms)  # graph build + first evaluation
    eng = model._engine
    calls = {"plain": lambda: eng.compute(), "peratom": lambda: eng.compute_peratom()}
    for _ in range(3):  # warm-up of both modes (the first per-atom call allocates its buffers)
        for f in calls.values():
            f()
    bwd = {k: [] for k in calls}
    wall = {k: [] for k in calls}
    for r in range(reps):
        for k in (("plain", "peratom") if r % 2 == 0 else ("peratom", "plain")):
            t0 = time.perf_counter()
            calls[k]()
            wall[k].append((time.perf_counter() - t0) * 1e3)
            bwd[k].append(eng.timings()["bwd_ms"])
    b0, b1 = np.median(bwd["plain"]), np.median(bwd["peratom"])
    print(f"{label} N {len(atoms)} reps {reps}: backward median plain {b0:.3f} ms (min {min(bwd['plain']):.3f} "
          f"max {max(bwd['plain']):.3f})  per-atom {b1:.3f} ms (min {min(bwd['peratom']):.3f} "
          f"max {max(bwd['peratom']):.3f})  +{(b1 / b0 - 1) * 100:.1f} %;  whole call median plain "
          f"{np.median(wall['plain']):.2f} ms  per-atom {np.median(wall['peratom']):.2f} ms", flush=True)
    eng.close()
