// kernels.cuh -- launch-side declarations of the CHGNet hot-path kernels (sm_100a).
//
// Formulation (verified against autograd in oracle/manual_ref.py):
//   first layer of every GatedMLP is split by input block, so the per-edge / per-angle work is
//     pre = gather(node projections) + (rank-9 radial term | dense 64->128 on the row's own feature)
//   followed by the 64x64 second layers, the gate product and a segmented sum.
// Reference arithmetic being replaced: SURVEY.md 8 rows a6-a15 (DistMLIP chgnet.py:208-453,
// chgnet_layers.py:16-119; matgl layer internals restated in SURVEY.md 9).
#pragma once
#include "common.cuh"

namespace b2m {

constexpr int TM = 128;   // rows (edges / angles) per tile
constexpr int LD = 132;   // smem row pitch of a [TM][128] tile (16B aligned, 4-bank skew)
constexpr int LDA = 68;   // smem row pitch of a [TM][64] tile
constexpr int NT = 256;   // threads per block for the fused tile kernels

struct RadialParams {
  float freq[NR];
  float rc;
  float norm;  // sqrt(2/rc)
  int p;
};

// -------- generic row GEMM: C[M,N] = (R | accum C | 0) + A[M,K] @ B[K,N] + bias --------
void launch_gemm(cudaStream_t st, const float* A, int lda, const float* B, float* C, int ldc, int M, int N, int K,
                 const float* bias, const float* R, int ldr, bool accum);

// -------- elementwise / init --------
void launch_embed(cudaStream_t st, int n, const int* type, const float* emb, float* x0);
void launch_bond_init(cudaStream_t st, int nb, const float4* b_vec, RadialParams rp, const float* W /*[64][9]*/,
                      float* out /*[nb,64]*/);
// Angle features (ang^l, and their adjoint gang) are touched only by the line-graph kernels, whose TMEM-imposed
// thread = row mapping makes every 16-byte access of a row-major [A][64] tensor its own L1 wavefront (LSU 49-63 % busy,
// profiles/r02k).  On the tcgen05 path they are therefore stored TILE-INTERLEAVED like the other kernel-private tensors:
//   float4 index ((tile * 16 + c/4) * 128 + r), tile = row / 128, r = row % 128   (a tile is one contiguous 32 KB block)
// The FP32-FFMA generation keeps row-major; `interleaved` selects the layout in the two kernels both paths share.
__host__ __device__ inline size_t ang_index(int64_t row, int c, int interleaved) {
  return interleaved ? ((size_t)((row >> 7) * 16 + (c >> 2)) * 128 + (size_t)(row & 127)) * 4 + (size_t)(c & 3)
                     : (size_t)row * 64 + (size_t)c;
}
void launch_angle_init(cudaStream_t st, int64_t na, const int* a_in, const int* a_out, const float4* b_vec,
                       const float* fa /*[5]*/, const float* Wae /*[64][9]*/, float* ang0, bool interleaved);
void launch_silu(cudaStream_t st, int64_t n, const float* pre, float* out);
void launch_dsilu_mul(cudaStream_t st, int64_t n, const float* pre, float* g);  // g *= dsilu(pre)
void launch_zero_rows(cudaStream_t st, float* p, int64_t nfloats);

// -------- atom conv (the edge-gather kernel of the headline metric) --------
struct AtomConvArgs {
  int64_t E;
  const int* e_src;
  const int* e_dst;
  const int* e_bond;
  const float4* e_vec;
  const float* Aproj;  // [n_loc,128]  x @ W1s^T
  const float* Cproj;  // [n_own,128]  x @ W1t^T + b1
  const float* Qproj;  // [B_own,128]  h @ W1e^T   (nullptr for layer 0)
  const float* M;      // [128][9]     W1e @ W_be
  const float* W2k;    // [2][64][64]  k-major second layers (L then G)
  const float* W2raw;  // [2][64][64]  as stored [out][in] (backward)
  const float* b2;     // [128]
  const float* Wabw;   // [64][9]
  RadialParams rp;
  // forward
  float* agg;  // [n_own,64] (+=)
  // backward
  const float* gagg;  // [n_own,64]
  float* gA;          // [n_loc,128] (+=, atomics)   nullptr -> skip (layer 0)
  float* gC;          // [n_own,128] (+=)
  float* gQ;          // [B_own,128] (=)
  float* gd;          // [E] (+=)
  // tcgen05 path: second-layer pre-activations (u | v) saved by the forward for the backward
  float* uv_save;       // [E,128] or nullptr (forward)
  const float* uv;      // [E,128] (backward)
  const float* be;      // [E,12] radial basis (9 used), computed once per step by launch_edge_basis
  const float* dbe;     // [E,12] d(be)/dd
};
void launch_edge_basis(cudaStream_t st, int64_t E, const float4* e_vec, RadialParams rp, float* be, float* dbe);
void launch_atomconv_fwd(cudaStream_t st, const AtomConvArgs& a);
void launch_atomconv_bwd(cudaStream_t st, const AtomConvArgs& a);

// -------- bond conv ("node" phase, HIDDEN) and angle update ("edge" phase, !HIDDEN) --------
struct LineArgs {
  int64_t A;
  const int* a_in;
  const int* a_out;
  const int* a_ctr;
  const float* ang;   // [A,64] input angle features
  const float* Ha;    // [B_loc,128]
  const float* Hb;    // [B_own,128] (+bias folded)
  const float* Xc;    // [n_loc,128]
  const float* Wgk;   // [2][64][64] k-major angle block of the first layer
  const float* Wgraw; // [128][64]   as stored (backward)
  const float* W2k;   // hidden only
  const float* W2raw;
  const float* b2;
  // forward outputs
  float* aggB;     // HIDDEN: [B_own,64] (+=)
  float* ang_out;  // !HIDDEN: [A,64]
  // backward
  const float* gaggB;  // HIDDEN: [B_own,64]
  float* gang;         // [A,64]: !HIDDEN reads it as upstream grad; both accumulate into it
  float* gHa;          // [B_loc,128] (+=)
  float* gHb;          // [B_own,128] (+=)
  float* gXc;          // [n_loc,128] (+=)
  // tcgen05 path: tensors saved by the forward for the backward
  float* uv_save;       // [A,128] last-layer pre-activations (u | v)
  float* ds_save;       // [A,128] silu'(first-layer pre-activation)   (HIDDEN only)
  const float* uv;
  const float* ds;
};
void launch_line_fwd(cudaStream_t st, const LineArgs& a, bool hidden);
void launch_line_bwd(cudaStream_t st, const LineArgs& a, bool hidden);

// -------- bond update: h' = h + upd * w3b(d_b) --------
void launch_bond_update_fwd(cudaStream_t st, int nb, const float4* b_vec, RadialParams rp3, const float* W3bw,
                            const float* h, const float* upd, float* hout);
// gupd = gh * w3b ; gdb += sum_k (sum_c gh*upd*W3bw[c][k]) * dtbe_k
void launch_bond_update_bwd(cudaStream_t st, int nb, const float4* b_vec, RadialParams rp3, const float* W3bw,
                            const float* gh, const float* upd, float* gupd, float* gdb);
// gdb += sum_k (sum_c gh0[b][c] Wbe[c][k]) dbe_k(d_b)
void launch_h0_bwd(cudaStream_t st, int nb, const float4* b_vec, RadialParams rp, const float* Wbe, const float* gh0,
                   float* gdb);
// theta / Fourier backward: gbvec[a], gbvec[b] += ...
void launch_angle_init_bwd(cudaStream_t st, int64_t na, const int* a_in, const int* a_out, const float4* b_vec,
                           const float* fa, const float* Wae, const float* gang0, float* gbvec, bool interleaved);

// -------- readout --------
// e_atom = y2 @ F2 + c2 (+elem ref); energy (double) += sum; site = x @ Ws + bs
void launch_rowdot(cudaStream_t st, int n, const float* X, const float* w, float bias, float* out, double* sum,
                   const int* type, const double* elem_ref, float scale);
// g[r][c] = scale * w[c] * dsilu(pre[r][c])
void launch_readout_seed(cudaStream_t st, int n, const float* pre, const float* w, float scale, float* g);
// per-atom energy of the owned rows, in global order: out[gid[i]] = scale * e_atom[i] + elem_ref[type[i]] + mean_per_atom
// (scale is the f32 data_std the energy sum uses, so that sum_i out[i] is the energy of the same evaluation)
void launch_atom_energy(cudaStream_t st, int n_own, const float* e_atom, const int* gid, const int* type,
                        const double* elem_ref, float scale, double mean_per_atom, double* out);

// -------- final geometry backward --------
// atom_vir: NULL (forces and total virial only), or [N][kAtomVirW] rows that also receive the per-atom virial
// (peratom.cuh); the per-atom instances leave forces and the total virial exactly as the plain ones compute them
constexpr int kAtomVirW = 12;
void launch_edge_final(cudaStream_t st, int64_t E, const int* e_src, const int* e_dst, const int* e_bond,
                       const float4* e_vec, const int* gid, const float* gd, const float* gdb, const float* gbvec,
                       float* forces /*[N,3]*/, double* virial /*[9]*/, float* atom_vir = nullptr);
void launch_halo_bond_final(cudaStream_t st, int b0, int b1, const int* b_src_gid, const int* b_dst,
                            const float4* b_vec, const int* gid, const float* gdb, const float* gbvec, float* forces,
                            double* virial, float* atom_vir = nullptr);

// -------- halo pack / unpack --------
void launch_gather_rows(cudaStream_t st, int n, int width, const int* idx, const float* src, float* dst);
void launch_scatter_add_rows(cudaStream_t st, int n, int width, const int* idx, const float* src, float* dst);

}  // namespace b2m

// ---------------------------------------------------------------------------------------------
// tcgen05 (5th-gen tensor core) variants.  3xTF32 split (hi*hi + lo*hi + hi*lo, fp32 accumulate in
// TMEM) keeps fp32-level accuracy.  Weights are pre-formatted on the host into the canonical
// K-major / no-swizzle core-matrix layout (8 rows x 16 B), hi and lo planes (see engine.cu: canon()).
// ---------------------------------------------------------------------------------------------
namespace b2m {
struct AtomConvTcW {
  const float* W2can;   // [4][4096]: W2L hi, W2L lo, W2G hi, W2G lo   (N=64, K=64)
  const float* Mcan;    // [2][2048]: M hi, M lo                        (N=128, K=16; k>=9 zero)
  const float* W2Tcan;  // [4][4096]: W2L^T hi, lo, W2G^T hi, lo        (backward: ghid = g . W2)
  int l2pf = 0;         // set by the launcher: prefetch the next tile's streamed blocks into L2
};
void launch_atomconv_fwd_tc(cudaStream_t st, const AtomConvArgs& a, const AtomConvTcW& w, int num_sms);
void launch_atomconv_bwd_tc(cudaStream_t st, const AtomConvArgs& a, const AtomConvTcW& w, int num_sms);
// third generation (kernels_ac3.cu): cp.async-staged gathers one tile ahead, no saved pre-activations unless uv_save
void launch_atomconv_fwd_v3(cudaStream_t st, const AtomConvArgs& a, const AtomConvTcW& w, int num_sms);
void launch_atomconv_bwd_v3(cudaStream_t st, const AtomConvArgs& a, const AtomConvTcW& w, int num_sms);
// C[M,N] = (R | accum C | 0) + A[M,K] @ B + bias, B given as canonical hi/lo planes of its [N][K] view.
// (K,N) in {(64,128), (64,64), (128,64)}.
void launch_gemm_tc(cudaStream_t st, const float* A, int lda, const float* Bcan, float* C, int ldc, int M, int N,
                    int K, const float* bias, const float* R, int ldr, bool accum, int num_sms);
// same kernel with an epilogue (TensorNet edge MLP): epi 1 keeps the pre-activation in Cpre (pitch ldc) and writes
// SiLU(value) to C; epi 2 multiplies the (accumulated) value by SiLU'(Pre[row][col]) (pitch ldp); epi 0 = plain
void launch_gemm_tc_epi(cudaStream_t st, const float* A, int lda, const float* Bcan, float* C, int ldc, int M, int N,
                        int K, const float* bias, bool accum, int epi, float* Cpre, const float* Pre, int ldp,
                        int num_sms);
struct LineTcW {
  const float* Wgcan;   // [2][8192]: first-layer angle block (N=128, K=64) hi, lo
  const float* W2can;   // [4][4096]: second layers (HIDDEN)
  const float* W2Tcan;  // [4][4096]: transposed second layers (HIDDEN, backward)
  const float* WgTcan;  // [4][4096]: per branch (N=64 angle cols, K=64 first-layer cols): L hi, L lo, G hi, G lo
  int l2pf = 0;         // set by the launcher: prefetch the next tile's streamed blocks into L2
};
void launch_line_fwd_tc(cudaStream_t st, const LineArgs& a, const LineTcW& w, bool hidden, int num_sms);
void launch_line_bwd_tc(cudaStream_t st, const LineArgs& a, const LineTcW& w, bool hidden, int num_sms);
}  // namespace b2m

// ---------------------------------------------------------------------------------------------
// TensorNet path (kernels_tn.cu).  Per-atom tensors in decomposed form [n][10][64] (I | a_xyz | S_xx xy xz yy yz zz).
// ---------------------------------------------------------------------------------------------
namespace b2m {
struct TnRadial {
  int nr;       // Gaussian centres in use
  int nrp;      // row pitch of the rbf / g_rbf buffers (multiple of 64, padding columns zero)
  float width;  // exp(-width (d - mu_k)^2)
  float rc;     // cosine cutoff radius
  float mu[64];
};
// C[z][M,N] = epi(A[z][M,K] @ B[K,N] + bias); z-batched over the 10 rows of a decomposed tensor when nz = 10
// (A + z*zA, C + z*zC, B = bsel ? (z==0 ? B0 : z<4 ? B1 : B2) : B0).  B is [K][N] row-major.  K % 32 == 0, N % 64 == 0.
// epi 0: store | 1: Cpre = value, C = SiLU(value) | 2: value *= SiLU'(Pre[m][n]) ; accum adds the old C afterwards.
struct TnGemm {
  const float* A = nullptr;
  int lda = 0;
  int64_t zA = 0;
  const float *B0 = nullptr, *B1 = nullptr, *B2 = nullptr;
  int bsel = 0;
  float* C = nullptr;
  int ldc = 0;
  int64_t zC = 0;
  float* Cpre = nullptr;
  const float* Pre = nullptr;
  int ldp = 0;
  const float* bias = nullptr;
  int M = 0, N = 0, K = 0, accum = 0, epi = 0;
};
void launch_tn_gemm(cudaStream_t st, const TnGemm& g, int nz);
void launch_tn_edge_geom(cudaStream_t st, int64_t E, const float4* e_vec, const TnRadial& rp, float* rbf, float* cut);
void launch_tn_embed_agg(cudaStream_t st, int n_own, const int* row_ptr, const int* e_src, const int* type,
                         const float* U, const float* V, const float* P, const float* cut, const float4* e_vec,
                         float* T0, float* nr0);
void launch_tn_layernorm(cudaStream_t st, int rows, int W, const float* x, const float* gamma, const float* beta,
                         float* y, float* stats);
void launch_tn_layernorm_bwd(cudaStream_t st, int rows, int W, const float* x, const float* stats, const float* gamma,
                             const float* gy, float* gx);
void launch_tn_embed_out(cudaStream_t st, int n, const float* T0m, const float* s2p, float* X0);
void launch_tn_embed_out_bwd(cudaStream_t st, int n, const float* T0m, const float* s2p, const float* gX0, float* gT0m,
                             float* gs2p);
void launch_tn_norm_bwd_add(cudaStream_t st, int n, const float* T0, const float* gnr0, float* gT0);
void launch_tn_embed_agg_bwd(cudaStream_t st, int64_t E, const int* e_src, const int* e_dst, const int* type,
                             const float* U, const float* V, const float* P, const float* cut, const float4* e_vec,
                             const float* gT0, float* gP, float* gC, float* gvh);
void launch_tn_scale(cudaStream_t st, int n, const float* X, float* Xh, float* q);
void launch_tn_scale_bwd(cudaStream_t st, int n, const float* X, const float* q, float* g);
void launch_tn_msg(cudaStream_t st, int n_own, const int* row_ptr, const int* e_src, const float* f3p, const float* cut,
                   const float* Y, float* msg);
void launch_tn_msg_bwd(cudaStream_t st, int n_own, const int* row_ptr, const int* e_src, const float* f3p,
                       const float* cut, const float* Y, const float* gmsg, float* g3, float* gC, float* gY);
void launch_tn_prod(cudaStream_t st, int n, const float* msg, const float* Y, int so3, float* Pn);
void launch_tn_prod_bwd(cudaStream_t st, int n, const float* msg, const float* Y, int so3, const float* gPn,
                        float* gmsg, float* gY);
void launch_tn_update(cudaStream_t st, int n, const float* Xh, const float* dX, float* Xn);
void launch_tn_update_bwd(cudaStream_t st, int n, const float* dX, const float* gXn, float* gdX);
void launch_tn_invariants(cudaStream_t st, int n, const float* X, float* inv);
void launch_tn_invariants_bwd(cudaStream_t st, int n, const float* X, const float* ginv, float* gX);
void launch_tn_readout_final(cudaStream_t st, int n, int W, const float* hL, const float* wL, float bL, const float* hG,
                             const float* wG, float bG, const int* type, const double* eref, float scale, float* lout,
                             float* gout, float* e_atom, double* energy);
void launch_tn_readout_seed(cudaStream_t st, int n, int W, const float* lout, const float* gout, float scale,
                            const float* wL, const float* wG, const float* preL, const float* preG, float* gL,
                            float* gG);
void launch_tn_edge_final(cudaStream_t st, int64_t E, const int* e_src, const int* e_dst, const float4* e_vec,
                          const int* gid, const TnRadial& rp, const float* g_rbf, const float* gC, const float* gvh,
                          float* gd, float* forces, double* virial, float* atom_vir = nullptr);
}  // namespace b2m
