"""ctypes binding of libb200mlip.so (the C-ABI in include/b200mlip.h).

There is NO CPU fallback: if the shared library is missing, or no sm_100 device is visible,
every entry point raises.  Nothing under oracle/ is ever imported from here.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200mlip.so")

SYMBOLS = [
    "b2m_create", "b2m_destroy", "b2m_last_error", "b2m_load_weights", "b2m_set_element_refs",
    "b2m_finalize_weights", "b2m_set_scaling", "b2m_comm_unique_id", "b2m_comm_init", "b2m_set_partition", "b2m_set_structure", "b2m_compute",
    "b2m_compute_resident", "b2m_get_sitewise", "b2m_get_counts", "b2m_get_partition_info",
    "b2m_debug_tensor", "b2m_last_timings", "b2m_release_workspace", "b2m_set_view", "b2m_create_tensornet",
    "b2m_compute_peratom",
]


class ModelDesc(C.Structure):
    _fields_ = [
        ("n_elem", C.c_int32), ("dim", C.c_int32), ("max_n", C.c_int32), ("max_f", C.c_int32),
        ("n_blocks", C.c_int32), ("cutoff_exponent", C.c_int32),
        ("cutoff", C.c_double), ("three_body_cutoff", C.c_double),
        ("data_mean", C.c_double), ("data_std", C.c_double),
    ]


class TensorNetDesc(C.Structure):
    _fields_ = [
        ("n_elem", C.c_int32), ("units", C.c_int32), ("num_rbf", C.c_int32), ("n_blocks", C.c_int32),
        ("so3", C.c_int32), ("reserved", C.c_int32),
        ("cutoff", C.c_double), ("rbf_width", C.c_double), ("data_mean", C.c_double), ("data_std", C.c_double),
    ]


class B2MError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libb200mlip error {code}: {msg}")
        self.code = code


_lib = None


def load_library():
    """dlopen the in-tree library and declare prototypes. Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -m distmlip_b200.build` "
            "(there is no CPU / PyTorch fallback for the CHGNet hot path)")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    vp, i32, i64, dbl = C.c_void_p, C.c_int, C.c_int64, C.c_double
    P = C.POINTER
    lib.b2m_create.argtypes = [P(ModelDesc), P(C.c_int), i32, P(vp)]
    lib.b2m_create_tensornet.argtypes = [P(TensorNetDesc), P(C.c_int), i32, P(vp)]
    lib.b2m_destroy.argtypes = [vp]
    lib.b2m_last_error.argtypes = [vp]
    lib.b2m_last_error.restype = C.c_char_p
    lib.b2m_load_weights.argtypes = [vp, C.c_char_p, P(C.c_float), P(i64), i32]
    lib.b2m_set_element_refs.argtypes = [vp, P(dbl), i32]
    lib.b2m_finalize_weights.argtypes = [vp]
    lib.b2m_set_scaling.argtypes = [vp, dbl, dbl]
    lib.b2m_comm_unique_id.argtypes = [C.c_char_p]
    lib.b2m_comm_init.argtypes = [vp, C.c_char_p, i32, i32]
    lib.b2m_set_partition.argtypes = [vp, i32, i32]
    lib.b2m_set_structure.argtypes = [vp, i64, P(dbl), P(dbl), P(C.c_int32), P(C.c_int), dbl]
    lib.b2m_compute.argtypes = [vp, i32, i32, P(dbl), P(C.c_float), P(C.c_float)]
    lib.b2m_compute_peratom.argtypes = [vp, i32, P(dbl), P(C.c_float), P(C.c_float), P(dbl), P(C.c_float)]
    lib.b2m_compute_resident.argtypes = [vp, i32, i32, i32, P(dbl), P(C.c_float)]
    lib.b2m_get_sitewise.argtypes = [vp, P(C.c_float)]
    lib.b2m_get_counts.argtypes = [vp, P(i64), i32]
    lib.b2m_get_partition_info.argtypes = [vp, i32, P(i64), i64]
    lib.b2m_get_partition_info.restype = i64
    lib.b2m_debug_tensor.argtypes = [vp, C.c_char_p, P(C.c_float), i64, P(i64), P(i64)]
    lib.b2m_last_timings.argtypes = [vp, P(dbl), i32]
    lib.b2m_release_workspace.argtypes = [vp]
    lib.b2m_set_view.argtypes = [vp, i32]
    for s in SYMBOLS:
        if s not in ("b2m_last_error", "b2m_get_partition_info"):
            getattr(lib, s).restype = C.c_int
    _lib = lib
    return lib


def comm_unique_id() -> bytes:
    lib = load_library()
    buf = C.create_string_buffer(128)
    rc = lib.b2m_comm_unique_id(buf)
    if rc != 0:
        raise B2MError(rc, (lib.b2m_last_error(None) or b"").decode())
    return buf.raw


class Engine:
    """Thin RAII wrapper over a b2m_handle.  `device`: one CUDA ordinal (one partition, or one rank of a multi-process
    job) or a list of ordinals = a single-process group with one partition per entry (ordinals may repeat)."""

    def __init__(self, *, n_elem, dim=64, max_n=9, max_f=4, n_blocks, cutoff, three_body_cutoff=0.0, cutoff_exponent=0,
                 data_mean=0.0, data_std=1.0, device=0, tensornet=None):
        """`tensornet`: None for CHGNet, else dict(units=, num_rbf=, so3=, rbf_width=) for a TensorNet handle
        (b2m_create_tensornet); everything after construction is the same."""
        self.lib = load_library()
        self.h = C.c_void_p()
        devs = [int(d) for d in device] if isinstance(device, (list, tuple)) else [int(device)]
        dev = (C.c_int * len(devs))(*devs)
        self.kind = "chgnet" if tensornet is None else "tensornet"
        if tensornet is None:
            self.desc = ModelDesc(n_elem, dim, max_n, max_f, n_blocks, cutoff_exponent, cutoff, three_body_cutoff,
                                  data_mean, data_std)
            rc = self.lib.b2m_create(C.byref(self.desc), dev, len(devs), C.byref(self.h))
        else:
            self.desc = TensorNetDesc(n_elem, int(tensornet["units"]), int(tensornet["num_rbf"]), n_blocks,
                                      int(bool(tensornet.get("so3", False))), 0, cutoff, float(tensornet["rbf_width"]),
                                      data_mean, data_std)
            rc = self.lib.b2m_create_tensornet(C.byref(self.desc), dev, len(devs), C.byref(self.h))
        if rc != 0:
            raise B2MError(rc, (self.lib.b2m_last_error(None) or b"").decode())
        self.natoms = 0
        self.rank, self.world = 0, len(devs)
        self.group = len(devs) > 1

    def _ck(self, rc):
        if rc != 0:
            raise B2MError(rc, (self.lib.b2m_last_error(self.h) or b"").decode())

    def close(self):
        if getattr(self, "h", None) is not None and self.h:
            self.lib.b2m_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- weights ----
    def load_state_dict(self, state_dict):
        for name, t in state_dict.items():
            a = np.ascontiguousarray(t.detach().cpu().numpy() if hasattr(t, "detach") else t, dtype=np.float32)
            if a.ndim == 0:
                a = a.reshape(1)
            shape = (C.c_int64 * a.ndim)(*a.shape)
            self._ck(self.lib.b2m_load_weights(self.h, name.encode(), a.ctypes.data_as(C.POINTER(C.c_float)), shape,
                                               a.ndim))

    def set_element_refs(self, offsets):
        """per-element energy offsets (double); None clears offsets set by an earlier Potential_Dist"""
        if offsets is None:
            self._ck(self.lib.b2m_set_element_refs(self.h, None, 0))
            return
        a = np.ascontiguousarray(offsets, dtype=np.float64)
        self._ck(self.lib.b2m_set_element_refs(self.h, a.ctypes.data_as(C.POINTER(C.c_double)), len(a)))

    def set_scaling(self, data_mean, data_std):
        self._ck(self.lib.b2m_set_scaling(self.h, float(data_mean), float(data_std)))

    def finalize(self):
        self._ck(self.lib.b2m_finalize_weights(self.h))

    def comm_init(self, unique_id: bytes | None, rank: int, world: int):
        self._ck(self.lib.b2m_comm_init(self.h, unique_id, rank, world))
        self.rank, self.world = rank, world

    def set_partition(self, rank: int, world: int):
        self._ck(self.lib.b2m_set_partition(self.h, rank, world))
        self.rank, self.world = rank, world

    # ---- structure / compute ----
    def set_structure(self, cart, lattice, species, pbc, tol=1e-8):
        """positions [n,3] f64 and species [n] i32 are handed to the library as they are (no copy when already contiguous
        in that dtype): it stages them through its own page-locked buffer with several copy threads"""
        cart = np.ascontiguousarray(cart, dtype=np.float64)
        species = np.ascontiguousarray(species, dtype=np.int32)
        n = len(cart)
        lattice = np.ascontiguousarray(lattice, dtype=np.float64).reshape(9)
        pbc = np.ascontiguousarray(pbc, dtype=np.int32)
        self.natoms = n
        self._ck(self.lib.b2m_set_structure(
            self.h, self.natoms, cart.ctypes.data_as(C.POINTER(C.c_double)),
            lattice.ctypes.data_as(C.POINTER(C.c_double)), species.ctypes.data_as(C.POINTER(C.c_int32)),
            pbc.ctypes.data_as(C.POINTER(C.c_int)), float(tol)))

    def compute(self, forces=True, stress=True, out_forces=None, out_stress=None):
        e = C.c_double()
        f = out_forces if out_forces is not None else (np.empty((self.natoms, 3), dtype=np.float32) if forces else None)
        s = out_stress if out_stress is not None else (np.empty(9, dtype=np.float32) if stress else None)
        fp = f.ctypes.data_as(C.POINTER(C.c_float)) if f is not None else None
        sp = s.ctypes.data_as(C.POINTER(C.c_float)) if s is not None else None
        self._ck(self.lib.b2m_compute(self.h, int(bool(forces)), int(bool(stress)), C.byref(e), fp, sp))
        return e.value, f, (s.reshape(3, 3) if s is not None else None)

    def compute_peratom(self, forces=True):
        """compute() plus per-atom output of the same evaluation: (E, F or None, stress [3,3] GPa, atom_e [N] eV,
        atom_W [N,3,3] eV).  sum(atom_e) == E and atom_W.sum(0) * 160.21766208 / V == stress (include/b200mlip.h)."""
        e = C.c_double()
        f = np.empty((self.natoms, 3), dtype=np.float32) if forces else None
        s = np.empty(9, dtype=np.float32)
        ae = np.empty(self.natoms, dtype=np.float64)
        aw = np.empty((self.natoms, 9), dtype=np.float32)
        fp = f.ctypes.data_as(C.POINTER(C.c_float)) if f is not None else None
        self._ck(self.lib.b2m_compute_peratom(self.h, int(bool(forces)), C.byref(e), fp,
                                              s.ctypes.data_as(C.POINTER(C.c_float)),
                                              ae.ctypes.data_as(C.POINTER(C.c_double)),
                                              aw.ctypes.data_as(C.POINTER(C.c_float))))
        return e.value, f, s.reshape(3, 3), ae, aw.reshape(-1, 3, 3)

    def compute_resident(self, reps=1, forces=True, stress=True):
        e = C.c_double()
        ms = C.c_float()
        self._ck(self.lib.b2m_compute_resident(self.h, int(bool(forces)), int(bool(stress)), int(reps), C.byref(e),
                                               C.byref(ms)))
        return e.value, ms.value

    def sitewise(self):
        out = np.empty(self.natoms, dtype=np.float32)
        self._ck(self.lib.b2m_get_sitewise(self.h, out.ctypes.data_as(C.POINTER(C.c_float))))
        return out

    def set_view(self, part):
        """single-process group: the partition that counts() / partition_info() describe"""
        self._ck(self.lib.b2m_set_view(self.h, int(part)))

    def counts(self, partition=None):
        if partition is not None:
            self.set_view(partition)
            try:
                return self.counts()
            finally:
                self.set_view(0)
        out = (C.c_int64 * 10)()
        self._ck(self.lib.b2m_get_counts(self.h, out, 10))
        keys = ["n_own", "n_halo", "n_edges", "n_bond_own", "n_bond_halo", "n_angles", "axis", "rank", "world",
                "launches"]
        return dict(zip(keys, [int(v) for v in out]))

    def partition_info(self, which):
        c = self.counts()
        cap = {0: c["n_own"], 1: c["n_halo"], 2: c["n_halo"], 3: 5 * c["n_edges"],
               4: 5 * (c["n_bond_own"] + c["n_bond_halo"]), 5: 3 * c["n_angles"], 6: 2 * c["n_own"] * 2 + 2,
               7: 16}[which]
        out = np.empty(max(cap, 1), dtype=np.int64)
        n = self.lib.b2m_get_partition_info(self.h, which, out.ctypes.data_as(C.POINTER(C.c_int64)), len(out))
        if n < 0:
            self._ck(int(n))
        out = out[:n]
        if which in (3, 4):
            return out.reshape(-1, 5)
        if which == 5:
            return out.reshape(-1, 3)
        if which == 6:
            return out.reshape(-1, 2)
        if which == 7:
            return out.view(np.float64)
        return out

    def debug_tensor(self, name):
        c = self.counts()
        cap = max(c["n_angles"], 3 * c["n_edges"], 10 * (c["n_own"] + c["n_halo"]), 1) * 64 + 64
        out = np.empty(cap, dtype=np.float32)
        r, k = C.c_int64(), C.c_int64()
        self._ck(self.lib.b2m_debug_tensor(self.h, name.encode(), out.ctypes.data_as(C.POINTER(C.c_float)), cap,
                                           C.byref(r), C.byref(k)))
        return out[: r.value * k.value].reshape(r.value, k.value).copy()

    def release_workspace(self):
        """free the resident graph and all per-structure device buffers (the next set_structure allocates again)"""
        self._ck(self.lib.b2m_release_workspace(self.h))

    def timings(self):
        out = (C.c_double * 5)()
        self._ck(self.lib.b2m_last_timings(self.h, out, 5))
        return dict(zip(["graph_ms", "fwd_ms", "bwd_ms", "edge_gather_ms", "total_ms"], [float(v) for v in out]))
