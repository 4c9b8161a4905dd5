"""Per-atom reference (test infrastructure): per-atom energies and virials of one f64 oracle evaluation
(oracle/chgnet_ref.py or oracle/tensornet_ref.py `potential_ref`), in the convention of b2m_compute_peratom
(include/b200mlip.h):

    e_i = data_std * e_atom_i + element_ref[type_i] + data_mean / N
    W_i = 1/2 sum_{e : src(e)=i or dst(e)=i} vec_e (x) dE/dvec_e        (eV, not symmetrised)

The oracles are used as they are.  In both, `vec` is the only path from positions and strain into `forward_graph` (pos
is otherwise unused), so retaining the gradient of the `vec` handed to `forward_graph` gives all of g_e = dE/dvec_e after
the oracle's own `backward()`; e_atom comes from the oracle's `e_atom` tap.  Then sum_i e_i = E and
sum_i W_i = dE/dstrain, i.e. sum_i W_i * 160.21766208 / V = the oracle's stress.
"""
from __future__ import annotations

import numpy as np
import torch

from oracle import chgnet_ref, tensornet_ref


def potential_ref_peratom(model, atoms, data_mean=0.0, data_std=1.0, element_refs=None, dtype=torch.float64,
                          **kw):
    """The oracle's (E, F, S[, site]) for `model` (a CHGNetRef or TensorNetRef) followed by (e_i [N], W_i [N,3,3])."""
    chgnet = isinstance(model, chgnet_ref.CHGNetRef)
    seen = {}
    inner = model.forward_graph

    def forward_graph(*args, **kwargs):
        # CHGNetRef.forward_graph(pos, vec, i1, i2, ..., node_types, taps) / TensorNetRef.forward_graph(vec, src, dst,
        # node_types, taps), both called positionally by potential_ref
        vec, i1, i2, types = (args[1], args[2], args[3], args[8]) if chgnet else (args[0], args[1], args[2], args[3])
        vec.retain_grad()
        seen.update(vec=vec, i1=i1, i2=i2, types=types)
        return inner(*args, **kwargs)

    taps = {}
    model.forward_graph = forward_graph
    try:
        ref = (chgnet_ref if chgnet else tensornet_ref).potential_ref(
            model, atoms, data_mean=data_mean, data_std=data_std, element_refs=element_refs, dtype=dtype, taps=taps,
            calc_forces=True, calc_stresses=True, **kw)
    finally:
        del model.forward_graph  # back to the class method
    vec, types = seen["vec"], seen["types"]
    n = types.shape[0]
    e_i = data_std * taps["e_atom"].detach().reshape(-1) + data_mean / n
    if element_refs is not None:
        e_i = e_i + torch.as_tensor(np.asarray(element_refs), dtype=e_i.dtype)[types]
    half = 0.5 * vec.detach()[:, :, None] * vec.grad[:, None, :]
    W = torch.zeros(n, 3, 3, dtype=half.dtype).index_add_(0, seen["i1"], half).index_add_(0, seen["i2"], half)
    return tuple(ref) + (e_i, W)
