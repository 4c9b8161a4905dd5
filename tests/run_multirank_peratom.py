"""Two-rank per-atom check, launched as
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tests/run_multirank_peratom.py
Every rank drives one GPU (NCCL halo exchange and all-reduce of the per-atom arrays inside libb200mlip); every rank must
hold the same per-atom energies and virials, equal to the single-partition oracle's and summing to the totals."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from distmlip_b200.implementations.matgl import CHGNet_Dist, Potential_Dist, TensorNet_Dist  # noqa: E402
from distmlip_b200.structures import SimpleAtoms, si_diamond  # noqa: E402
from tests._util import make_model  # noqa: E402
from tests.peratom_ref import potential_ref_peratom  # noqa: E402
from tests.test_oracle_tensornet import make_tn  # noqa: E402

GPA_PER_EVA3 = 160.21766208


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ok = True
    a0 = si_diamond(3, nz=4 * world, seed=9)
    atoms = SimpleAtoms(["O" if i % 3 == 0 else "Si" for i in range(len(a0))], a0.get_positions(), a0.get_cell())
    for kind in ("chgnet", "tensornet"):
        model = make_model() if kind == "chgnet" else make_tn(seed=3, scale=1.5)
        refs = np.linspace(-3.0, -1.0, len(model.element_types))
        dm = (CHGNet_Dist if kind == "chgnet" else TensorNet_Dist).from_existing(model)
        dm.enable_distributed_mode(list(range(world)))
        pot = Potential_Dist(model=dm, data_mean=0.7, data_std=1.3, element_refs=refs, calc_per_atom=True)
        E, F, S, _ = pot(atoms)
        ae, st = pot.last_dist_info.energies, pot.last_dist_info.stresses
        de_sum = abs(ae.sum() - E.item())
        ds_sum = np.abs(st.sum(0) - S.numpy()).max()
        ok = ok and de_sum < 1e-9 * abs(E.item()) and ds_sum < 1e-5 * np.abs(st).sum(0).max() + 1e-7
        if rank == 0:
            ref = potential_ref_peratom(model.double(), atoms, data_mean=0.7, data_std=1.3, element_refs=refs)
            eo, Wo = ref[-2].numpy(), ref[-1].numpy()
            de = np.abs(ae - eo).max()
            dw = np.abs(st * atoms.get_volume() / GPA_PER_EVA3 - Wo).max()
            print(f"{kind} world {world} natoms {len(atoms)}: max|de_i| {de:.2e} max|dW_i| {dw:.2e} "
                  f"(max|W| {np.abs(Wo).max():.2e}) |sum e - E| {de_sum:.1e} |sum s - S| {ds_sum:.1e}", flush=True)
            ok = ok and de < 1e-5 and dw < 1e-5 * np.abs(Wo).max() + 1e-6
        # all ranks must hold identical (all-reduced) per-atom arrays
        t = torch.tensor(np.concatenate([ae, st.ravel()]), device="cuda")
        tmax, tmin = t.clone(), t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
        ok = ok and float((tmax - tmin).abs().max()) == 0.0
        dm._engine.close()
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("MULTIRANK PERATOM", "PASS" if flag.item() == 1 else "FAIL", flush=True)
    dist.destroy_process_group()
    sys.exit(0 if flag.item() == 1 else 1)


if __name__ == "__main__":
    main()
