/*
 * b200mlip.h -- C-ABI of libb200mlip.so: the B200-native (sm_100a) engine behind the
 * DistMLIP-compatible CHGNet hot path.  Plain C, no CPython / NumPy / torch types.
 *
 * What each entry point replaces in the reference (AegisIK/DistMLIP @ 9824cd4):
 *
 *   b2m_create / b2m_load_weights / b2m_finalize_weights
 *        CHGNet_Dist.from_existing + enable_distributed_mode, which deep-copy every sub-module
 *        onto every GPU (DistMLIP/implementations/matgl/models/chgnet.py:455-560).
 *   b2m_set_structure
 *        Distributed.create_distributed -> get_subgraphs_fast, the CPU neighbour list + slab
 *        partitioner + bond/line-graph builder run on every calculate()
 *        (DistMLIP/distributed/dist.py:158-275; subgraph_creation_fast.c:92-453; fpis.c:418-901;
 *        subgraph_creation_utils.c:26-931), plus the geometry block of potential_forward_dist
 *        (chgnet.py:33-197).
 *   b2m_compute
 *        CHGNet_Dist.dist_forward (chgnet.py:208-453) + Potential_Dist.forward's scaling,
 *        torch.autograd.backward, F = -grad, sigma = strain.grad / V * 160.21766208
 *        (DistMLIP/implementations/matgl/pes.py:50-146).
 *   b2m_create with ndev > 1, or b2m_comm_unique_id / b2m_comm_init
 *        the reference has no communicator: Distributed.transfer_nodes does cross-device
 *        slice copies from one thread (dist.py:323-358).  Here either one process drives every
 *        GPU (ndev > 1: peer-memory halo stores ordered by CUDA events, one host thread per
 *        partition) or one process per GPU with NCCL point-to-point halo exchange between slab
 *        neighbours.
 *   b2m_get_partition_info
 *        the 19-tuple returned by get_subgraphs_fast (subgraph_creation_fast.c:403-422), in
 *        canonical (set) form, for parity tests.
 *
 * Conventions: every call returns 0 on success, <0 on error (message via b2m_last_error);
 * the library never calls exit().  Caller owns all host buffers; the library owns all device
 * memory, streams and NCCL communicators.  A handle is single-caller (no internal locking) and
 * may be used with the GIL released.
 */
#ifndef B200MLIP_H
#define B200MLIP_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct b2m_engine* b2m_handle;

/* error codes */
#define B2M_OK 0
#define B2M_ERR_INVALID (-1)     /* bad argument / unsupported model dimension          */
#define B2M_ERR_PARTITIONS (-2)  /* num_partitions < 1                                   */
#define B2M_ERR_SELF_EDGE (-3)   /* unused: periodic self images are never neighbours    */
#define B2M_ERR_SLAB_WIDTH (-4)  /* slab width <= 2 (r_cut [+ r_bond])  (ref: utils.c:1512-1529) */
#define B2M_ERR_CUDA (-5)        /* CUDA / NCCL runtime failure                          */
#define B2M_ERR_STATE (-6)       /* call order violation (e.g. compute before set_structure) */

typedef struct {
  int32_t n_elem;            /* rows of atom_embedding.weight                      */
  int32_t dim;               /* atom = bond = angle feature width (64 supported)   */
  int32_t max_n;             /* radial basis size (9 supported)                    */
  int32_t max_f;             /* Fourier order (4 supported -> 9 features)          */
  int32_t n_blocks;          /* number of atom-graph blocks (>= 2)                 */
  int32_t cutoff_exponent;   /* polynomial envelope exponent p                     */
  double cutoff;             /* r_cut  (Angstrom)                                  */
  double three_body_cutoff;  /* r_bond (Angstrom)                                  */
  double data_mean;          /* Potential: E = std * E + mean (pes.py:109)         */
  double data_std;
} b2m_model_desc;

/* devices: CUDA ordinals owned by this handle, one per partition (SURVEY 8b; the reference's
 * enable_distributed_mode(gpus), chgnet.py:455-549).
 *   ndev == 1: one partition, or one rank of a multi-process job (b2m_comm_init).
 *   ndev  > 1: a single-process group: partition p runs on devices[p] (ordinals may repeat, e.g.
 *              {0, 0} = two partitions on one GPU), one host thread + stream per partition inside
 *              b2m_set_structure / b2m_compute, halo rows exchanged as direct peer-memory stores
 *              ordered by CUDA events (no NCCL).  b2m_get_counts / b2m_get_partition_info describe
 *              the partition chosen with b2m_set_view (default 0), b2m_debug_tensor partition 0;
 *              energies, forces, stress and the site-wise readout are those of the whole structure. */
int b2m_create(const b2m_model_desc* desc, const int* devices, int ndev, b2m_handle* out);
int b2m_destroy(b2m_handle h);
const char* b2m_last_error(b2m_handle h);

/* TensorNet (SURVEY.md 8(f).2): the same handle type and every call below, for a model with matgl's TensorNet attribute
 * tree (DistMLIP/implementations/matgl/models/tensornet.py:163-204: bond_expansion, tensor_embedding, layers, out_norm,
 * linear, final_layer).  Supported: units = 64, Gaussian bond expansion (<= 64 centres), swish, O(3) or SO(3),
 * is_intensive = False, no state features.  No bond graph: use_bond_graph False, three_body_cutoff 0 (pes.py:79-80).
 * b2m_get_sitewise is an error on such a handle. */
typedef struct {
  int32_t n_elem;    /* len(element_types)                                            */
  int32_t units;     /* 64                                                            */
  int32_t num_rbf;   /* Gaussian centres (the centres themselves are a state_dict key) */
  int32_t n_blocks;  /* interaction layers                                            */
  int32_t so3;       /* equivariance_invariance_group: 0 = "O(3)", 1 = "SO(3)"       */
  int32_t reserved;
  double cutoff;     /* r_cut (Angstrom), also the cosine cutoff radius               */
  double rbf_width;  /* exp(-width (d - mu)^2)                                        */
  double data_mean;
  double data_std;
} b2m_tensornet_desc;
int b2m_create_tensornet(const b2m_tensornet_desc* desc, const int* devices, int ndev, b2m_handle* out);

/* One call per state_dict key of the matgl CHGNet attribute tree (SURVEY.md 8c), fp32 row-major. */
int b2m_load_weights(b2m_handle h, const char* name, const float* host_ptr, const int64_t* shape, int ndim);
/* Optional per-element energy offsets (Potential.element_refs), length n_elem. */
int b2m_set_element_refs(b2m_handle h, const double* offsets, int n);
/* Potential scaling E = std * E + mean (pes.py:109); may be changed between computes. */
int b2m_set_scaling(b2m_handle h, double data_mean, double data_std);
/* Composes derived matrices, uploads everything. Fails if a required key is missing. */
int b2m_finalize_weights(b2m_handle h);

/* Multi-process graph parallelism: rank 0 makes an id, every rank calls b2m_comm_init with it. */
int b2m_comm_unique_id(char* out128);
int b2m_comm_init(b2m_handle h, const char* id128, int rank, int world);
/* Graph-only view of partition `rank` of `world` without a communicator (parity tests of the
 * partitioner on one GPU).  b2m_compute refuses to run in this state when world > 1. */
int b2m_set_partition(b2m_handle h, int rank, int world);

/* Graph build (neighbour list, slab partition, halo sections, bond graph, angles) on the GPU.
 * cart: [natoms,3] f64 Cartesian (unwrapped ok); lattice9: row vectors; species: index into
 * element_types; pbc3: 0/1 flags.  tol as in the reference (1e-8 on d^2). */
int b2m_set_structure(b2m_handle h, int64_t natoms, const double* cart, const double* lattice9,
                      const int32_t* species, const int* pbc3, double tol);

/* Energy (+forces [natoms,3] eV/A, +stress [9] GPa).  forces/stress9 may be NULL.
 * With world > 1 every rank receives the full (all-reduced) result. */
int b2m_compute(b2m_handle h, int want_forces, int want_stress, double* energy, float* forces, float* stress9);
/* b2m_compute (energy, forces if want_forces, stress) plus per-atom output of the same evaluation.  CHGNet and
 * TensorNet handles, every process model; atom_energy / atom_virial9 may be NULL.  For N atoms and cell volume V:
 *   atom_energy [natoms] f64, eV:   e_i = data_std * e^_i + element_ref[type_i] + data_mean / N
 *        (e^_i: the model's raw per-atom output); sum_i e_i = energy of the same call.
 *   atom_virial9 [natoms,9] f32, eV, row-major 3x3, not symmetrised:
 *        W_i[a][b] = 1/2 sum_{e : src(e)=i or dst(e)=i} vec_e[a] g_e[b],
 *        vec_e = x_dst + off.L - x_src, g_e = dE/dvec_e (each edge's term split evenly between its two atoms);
 *        sum_i W_i = dE/dstrain, so sum_i W_i * 160.21766208 / V = stress9 (GPa) of the same call.
 * The per-atom buffers (56 B per atom and partition) are allocated by the first such call. */
int b2m_compute_peratom(b2m_handle h, int want_forces, double* energy, float* forces, float* stress9,
                        double* atom_energy /* [natoms] or NULL */, float* atom_virial9 /* [natoms,9] eV or NULL */);
/* Same arithmetic, graph already resident; runs `reps` passes and returns device time (ms) of
 * the last one measured with CUDA events on the compute stream. Used by bench.py `value`. */
int b2m_compute_resident(b2m_handle h, int want_forces, int want_stress, int reps, double* energy, float* ms);

/* site-wise readout (magmom) for all atoms, [natoms] */
int b2m_get_sitewise(b2m_handle h, float* out);

/* Single-process groups: which partition b2m_get_counts / b2m_get_partition_info describe (default 0).  The reference's
 * Distributed keeps every partition's arrays on the host (dist.py:39-99) and its counters take a `partition` argument
 * (dist.py:462-551); this is the equivalent view. */
int b2m_set_view(b2m_handle h, int part);

/* counts: [0]=n_own [1]=n_halo [2]=n_edges [3]=n_bond_own [4]=n_bond_halo [5]=n_angles
 *         [6]=partition axis [7]=rank [8]=world [9]=kernel launches in last compute */
int b2m_get_counts(b2m_handle h, int64_t* out, int n);

/* Partition info export (int64, canonical content; see DESIGN.md "partition export"):
 *   which = 0: owned atom gids                 [n_own]
 *           1: halo atom gids                  [n_halo]   (grouped by owner, gid ascending)
 *           2: halo owner partition            [n_halo]
 *           3: edges (src gid, dst gid, ox,oy,oz)        [n_edges,5]
 *           4: bonds (src gid, dst gid, ox,oy,oz), owned first then halo  [n_bond,5]
 *           5: angles (in-bond id, out-bond id, centre gid)               [n_angles,3]
 *           6: to-lists (q, gid) pairs          [n_to,2]
 *           7: walls as IEEE-754 bit patterns   [world-1]
 * Returns number of int64 written, or <0. cap = capacity of out in int64 elements. */
int64_t b2m_get_partition_info(b2m_handle h, int which, int64_t* out, int64_t cap);

/* Debug taps (tests only): copies a named device tensor to host (fp32). rows/cols returned. */
int b2m_debug_tensor(b2m_handle h, const char* name, float* out, int64_t cap, int64_t* rows, int64_t* cols);

/* Frees the resident graph and every per-structure device buffer (weights, streams and communicators stay); the next
 * b2m_set_structure allocates again.  For callers that want the memory back between structures of very different size. */
int b2m_release_workspace(b2m_handle h);

/* Per-phase device timings (ms) of the last b2m_compute: [0]=graph build [1]=forward [2]=backward
 * [3]=edge-gather (atom conv fwd) kernel average [4]=total */
int b2m_last_timings(b2m_handle h, double* out, int n);

#ifdef __cplusplus
}
#endif
#endif
