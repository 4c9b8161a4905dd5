"""GPU: per-atom energies and virials (b2m_compute_peratom) of CHGNet and TensorNet against the f64 oracles
(tests/peratom_ref.py over oracle/chgnet_ref.py and oracle/tensornet_ref.py), their sum rules against the totals of the same call,
partition independence in single-process groups, and the ASE surface.

Tolerances (f32 engine vs f64 oracle): |de_i| <= 1e-5 eV and |dW_i| <= 1e-5 max|W| + 1e-6 eV.  Each test prints what it
observed; on a B200 the largest errors were 1.0e-7 eV in e_i and 2.2e-7 eV in W_i (max|W| ~ 0.1 eV), so the bounds
leave about two orders of magnitude of margin for other weights and structures."""
import numpy as np
import pytest
import torch

from distmlip_b200.structures import SimpleAtoms, rough_cell, si_diamond
from tests._util import engine_from_model, make_model
from tests.peratom_ref import potential_ref_peratom
from tests.test_gpu_tensornet import tn_engine
from tests.test_oracle_tensornet import make_tn, tn_graph

pytestmark = pytest.mark.gpu
GPA_PER_EVA3 = 160.21766208
MEAN, STD = 0.7, 1.3
TOL_E, TOL_W_REL, TOL_W_ABS = 1e-5, 1e-5, 1e-6


def mixed(atoms, other="O", every=3):
    sym = [other if i % every == 0 else s for i, s in enumerate(atoms.get_chemical_symbols())]
    return SimpleAtoms(sym, atoms.get_positions(), atoms.get_cell())


def refs_for(model):
    return np.linspace(-3.0, -1.0, len(model.element_types))


def set_structure(eng, model, atoms):
    sp = np.array([model.element_types.index(s) for s in atoms.get_chemical_symbols()], dtype=np.int32)
    eng.set_structure(atoms.get_positions(), np.array(atoms.get_cell()), sp, atoms.get_pbc().astype(np.int32))


def check_sum_rules(atoms, E, S, ae, aw):
    n = len(atoms)
    assert ae.shape == (n,) and aw.shape == (n, 3, 3)
    de = abs(ae.sum() - E)
    assert de < 1e-9 * max(1.0, abs(E)), de
    Ssum = aw.astype(np.float64).sum(0) * GPA_PER_EVA3 / atoms.get_volume()
    scale = np.abs(aw).astype(np.float64).sum(0).max() * GPA_PER_EVA3 / atoms.get_volume()
    ds = np.abs(Ssum - S).max()
    assert ds < 1e-5 * scale + 1e-7, (ds, scale)
    return de, ds


def check_vs_oracle(label, atoms, got, ref):
    E, _F, S, ae, aw = got
    Eo, eo, Wo = float(ref[0]), ref[-2].numpy(), ref[-1].numpy()
    de = np.abs(ae - eo).max()
    dw = np.abs(aw - Wo).max()
    wmax = np.abs(Wo).max()
    sde, sds = check_sum_rules(atoms, E, S, ae, aw)
    print(f"{label}: N {len(atoms)} max|de_i| {de:.2e} eV  max|dW_i| {dw:.2e} eV (max|W| {wmax:.2e})  "
          f"|sum e - E| {sde:.1e}  |sum W/V - S| {sds:.1e} GPa  |E - E_oracle| {abs(E - Eo):.1e}")
    assert de <= TOL_E, de
    assert dw <= TOL_W_REL * wmax + TOL_W_ABS, (dw, wmax)


# ------------------------------------------------------------------ CHGNet
@pytest.fixture(scope="module")
def chg():
    m = make_model()
    eng = engine_from_model(m, data_mean=MEAN, data_std=STD, element_refs=refs_for(m))
    yield m, eng
    eng.close()


def chg_oracle(atoms):
    m = make_model().double()
    return potential_ref_peratom(m, atoms, data_mean=MEAN, data_std=STD, element_refs=refs_for(m))


CHG_CASES = {
    "diamond64": lambda: mixed(si_diamond(2, seed=1)),
    "diamond512": lambda: mixed(si_diamond(4, seed=2)),
    "diamond8000": lambda: mixed(si_diamond(10, seed=31)),
    "rough2400": lambda: mixed(rough_cell(2400, seed=5, aspect=(1, 1, 4))),
}


@pytest.mark.parametrize("case", list(CHG_CASES))
def test_chgnet_per_atom_matches_oracle(chg, case):
    m, eng = chg
    atoms = CHG_CASES[case]()
    set_structure(eng, m, atoms)
    check_vs_oracle(f"chgnet {case}", atoms, eng.compute_peratom(), chg_oracle(atoms))


def test_chgnet_totals_unchanged(chg):
    m, eng = chg
    atoms = CHG_CASES["rough2400"]()
    set_structure(eng, m, atoms)
    E0, F0, S0 = eng.compute()
    E1, F1, S1, _ae, _aw = eng.compute_peratom()
    E2, F2, S2 = eng.compute()  # a plain evaluation after a per-atom one
    n = len(atoms)
    for E, F, S in ((E1, F1, S1), (E2, F2, S2)):
        assert abs(E - E0) / n < 2e-8
        assert np.abs(F - F0).max() <= 1e-5 * np.abs(F0).max()
        assert np.abs(S - S0).max() <= 1e-5 * np.abs(S0).max()
    _e, f_none, s3, ae3, _aw3 = eng.compute_peratom(forces=False)
    assert f_none is None and abs(ae3.sum() - E0) / n < 2e-8


@pytest.mark.parametrize("nparts", [2, 3])
def test_chgnet_group_reproduces_one_partition(chg, nparts):
    m, one = chg
    atoms = mixed(si_diamond(4, nz=4 * nparts, seed=3))  # 21.7 A slabs > 2 (r_cut + r_bond)
    set_structure(one, m, atoms)
    E1, _F1, S1, ae1, aw1 = one.compute_peratom()
    grp = engine_from_model(m, device=[0] * nparts, data_mean=MEAN, data_std=STD, element_refs=refs_for(m))
    set_structure(grp, m, atoms)
    assert grp.counts()["n_halo"] > 0
    E2, _F2, S2, ae2, aw2 = grp.compute_peratom()
    check_sum_rules(atoms, E2, S2, ae2, aw2)
    de, dw = np.abs(ae2 - ae1).max(), np.abs(aw2 - aw1).max()
    print(f"chgnet group {nparts}: max|de_i| {de:.2e}  max|dW_i| {dw:.2e} (max|W| {np.abs(aw1).max():.2e})")
    assert de < 5e-6 and dw <= 1e-5 * np.abs(aw1).max() + 1e-7
    grp.close()


def test_chgnet_perfect_diamond_is_uniform(chg):
    m, eng = chg
    atoms = si_diamond(4, sigma=0)
    set_structure(eng, m, atoms)
    _E, _F, _S, ae, aw = eng.compute_peratom()
    de = np.abs(ae - ae.mean()).max()
    dw = np.abs(aw - aw.mean(0)).max()
    print(f"chgnet perfect diamond: spread e_i {de:.2e} (|e| {abs(ae.mean()):.2e})  spread W_i {dw:.2e} "
          f"(max|W| {np.abs(aw.mean(0)).max():.2e})")
    assert de <= 2e-6 * abs(ae.mean()) + 1e-6
    assert dw <= 1e-5 * np.abs(aw.mean(0)).max() + 1e-7


# ------------------------------------------------------------------ TensorNet
def tn_case(group):
    m = make_tn(seed=3, scale=1.5, equivariance_invariance_group=group)
    return m


def tn_oracle(m, atoms):
    og = tn_graph(atoms, float(m.cutoff))
    return potential_ref_peratom(m, atoms, graph=(og["i1"], og["i2"], og["off"]), data_mean=MEAN, data_std=STD,
                                 element_refs=refs_for(m))


@pytest.mark.parametrize("group", ["O(3)", "SO(3)"])
@pytest.mark.parametrize("parts", [1, 2])
def test_tensornet_per_atom_matches_oracle(group, parts):
    m = tn_case(group)
    eng = tn_engine(m, device=[0] * parts if parts > 1 else 0, data_mean=MEAN, data_std=STD,
                    element_refs=refs_for(m))
    for label, atoms in (("diamond", mixed(si_diamond(2, seed=3, nz=4 * parts))),
                         ("rough", mixed(rough_cell(300 * parts, seed=4, aspect=(1, 1, parts))))):
        set_structure(eng, m, atoms)
        got = eng.compute_peratom()
        check_vs_oracle(f"tensornet {group} parts {parts} {label}", atoms, got, tn_oracle(m, atoms))
        E0, F0, S0 = eng.compute()
        assert abs(E0 - got[0]) / len(atoms) < 2e-6
    eng.close()


def test_tensornet_perfect_diamond_is_uniform():
    m = tn_case("O(3)")
    eng = tn_engine(m, data_mean=MEAN, data_std=STD)
    atoms = si_diamond(3, sigma=0)
    set_structure(eng, m, atoms)
    _E, _F, _S, ae, aw = eng.compute_peratom()
    de = np.abs(ae - ae.mean()).max()
    dw = np.abs(aw - aw.mean(0)).max()
    print(f"tensornet perfect diamond: spread e_i {de:.2e}  spread W_i {dw:.2e} (max|W| {np.abs(aw.mean(0)).max():.2e})")
    assert de <= 2e-6 * abs(ae.mean()) + 1e-6
    assert dw <= 1e-5 * np.abs(aw.mean(0)).max() + 1e-7
    eng.close()


# ------------------------------------------------------------------ Python / ASE surface
@pytest.mark.parametrize("devices", [[0], [0, 0]])
def test_ase_calculator_per_atom_on_the_engine(devices):
    from distmlip_b200.implementations.matgl import CHGNet_Dist, PESCalculator_Dist, Potential_Dist

    m = make_model()
    dm = CHGNet_Dist.from_existing(m)
    dm.enable_distributed_mode(devices)
    pot = Potential_Dist(model=dm, data_mean=MEAN, data_std=STD, element_refs=refs_for(m), calc_per_atom=True)
    atoms = mixed(si_diamond(3, nz=8, seed=6))
    calc = PESCalculator_Dist(potential=pot, stress_weight=0.5)
    calc.calculate(atoms, ["energy", "forces", "stress", "energies", "stresses"])
    r = calc.results
    n = len(atoms)
    assert r["energies"].shape == (n,) and r["stresses"].shape == (n, 3, 3)
    assert abs(r["energies"].sum() - r["energy"]) < 1e-9 * abs(r["energy"])
    scale = np.abs(r["stresses"]).sum(0).max()
    assert np.abs(r["stresses"].sum(0) - r["stress"]).max() < 1e-5 * scale + 1e-7
    ref = chg_oracle(atoms)
    assert np.abs(r["energies"] - ref[-2].numpy()).max() < TOL_E
    info = pot.last_dist_info
    assert np.allclose(info.stresses * 0.5, r["stresses"])
    dm._engine.close()


# ------------------------------------------------------------------ one process per GPU (NCCL)
def test_two_rank_per_atom():
    import os
    import subprocess
    import sys

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", "29557", os.path.join(root, "tests", "run_multirank_peratom.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=root)
    assert r.returncode == 0 and "MULTIRANK PERATOM PASS" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
