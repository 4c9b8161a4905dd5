import os, sys, time, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from distmlip_b200.structures import si_diamond
from tests._util import make_model, engine_from_model
m = make_model(); eng = engine_from_model(m)
for world in (1, 2, 4, 8):
    atoms = si_diamond(23, nz=23*world)
    cart, lat = atoms.get_positions(), atoms.get_cell()
    spec = np.zeros(len(atoms), dtype=np.int32); pbc = np.ones(3, dtype=np.int32)
    for rank in sorted({0, world//2}):
        eng.set_partition(rank, world)
        for it in range(3):
            t0 = time.perf_counter(); eng.set_structure(cart, lat, spec, pbc); dt = time.perf_counter()-t0
        c = eng.counts()
        print(f"world {world} rank {rank} N {len(atoms)} wall {dt*1e3:.2f} ms graph_ms {eng.timings()['graph_ms']:.2f} own {c['n_own']} halo {c['n_halo']}", flush=True)
eng.set_partition(0,1)
