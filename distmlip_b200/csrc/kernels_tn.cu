// kernels_tn.cu -- TensorNet (O(3)-equivariant Cartesian-tensor message passing) on the same partitioned CSR graph as
// the CHGNet path.  SURVEY.md 8(f).2; replaces the matgl / DGL arithmetic behind
// DistMLIP/implementations/matgl/models/tensornet.py:10-161 (layer internals: matgl TensorEmbedding,
// TensorNetInteraction, WeightedReadOut -- restated in oracle/tensornet_ref.py, staged exactly as here in
// oracle/tensornet_manual.py).
//
// Storage: a per-atom, per-channel 3x3 tensor M = I*eye + skew(a) + S is held in "decomposed form" as 10 rows of
// C = 64 channels, [n][10][64]:  0: I | 1..3: a_x a_y a_z | 4..9: S_xx S_xy S_xz S_yy S_yz S_zz.  The channel mixes
// (linears_tensor) act on each of the 10 rows with the weight of its part, so they are one z-batched row GEMM; the
// element-wise tensor algebra is one thread per (atom, channel), coalesced over channels; aggregations walk the
// CSR-by-destination rows (no atomics in the forward); the reverse pass scatters to sources with red.add.
// First generation of this path.  The edge-level products (edge MLP 32 -> 64 -> 128 -> 192 and the three distance
// projections, 49 % of a step) run on the tcgen05 row GEMM of the CHGNet path (kernels_tc.cu, k_gemm_tc_pipe with a
// SiLU / SiLU' epilogue; engine_tn.inl composes the 192-wide layers from its 64/128 shapes); the node-level products
// (channel mixes, scalar MLPs, readout) use the FP32-FFMA tile kernel below, which also serves the edge level under
// B2M_TN_FFMA=1 (A/B checks).  DESIGN.md 8 lists what comes next.
#include <math_constants.h>

#include "kernels.cuh"
#include "peratom.cuh"

namespace b2m {

namespace {

constexpr int TC = 64;        // channels
constexpr int TW = 10 * TC;   // floats per atom in decomposed form

__device__ __forceinline__ int part_of(int k) { return k == 0 ? 0 : (k < 4 ? 1 : 2); }
__device__ __forceinline__ float nw_of(int k) {  // tensor_norm = sum_k nw[k] t_k^2
  return k == 0 ? 3.f : ((k < 4 || k == 5 || k == 6 || k == 8) ? 2.f : 1.f);
}
__device__ __forceinline__ float sigm(float x) { return 1.f / (1.f + __expf(-x)); }
__device__ __forceinline__ float silu_f(float x) { return x * sigm(x); }
__device__ __forceinline__ float dsilu_f(float x) {
  const float s = sigm(x);
  return s * (1.f + x * (1.f - s));
}

__device__ __forceinline__ void full9(const float* t, float* m) {
  m[0] = t[0] + t[4], m[1] = t[5] - t[3], m[2] = t[6] + t[2];
  m[3] = t[5] + t[3], m[4] = t[0] + t[7], m[5] = t[8] - t[1];
  m[6] = t[6] - t[2], m[7] = t[8] + t[1], m[8] = t[0] + t[9];
}
__device__ __forceinline__ void full_adj(const float* g, float* t) {  // dE/dM -> parameter space
  t[0] = g[0] + g[4] + g[8];
  t[1] = g[7] - g[5], t[2] = g[2] - g[6], t[3] = g[3] - g[1];
  t[4] = g[0], t[5] = g[1] + g[3], t[6] = g[2] + g[6], t[7] = g[4], t[8] = g[5] + g[7], t[9] = g[8];
}
__device__ __forceinline__ void dec10(const float* m, float* t) {
  const float I = (m[0] + m[4] + m[8]) * (1.f / 3.f);
  t[0] = I;
  t[1] = 0.5f * (m[7] - m[5]), t[2] = 0.5f * (m[2] - m[6]), t[3] = 0.5f * (m[3] - m[1]);
  t[4] = m[0] - I, t[5] = 0.5f * (m[1] + m[3]), t[6] = 0.5f * (m[2] + m[6]);
  t[7] = m[4] - I, t[8] = 0.5f * (m[5] + m[7]), t[9] = m[8] - I;
}
__device__ __forceinline__ void dec_adj(const float* g, float* G) {
  const float t = (g[0] - g[4] - g[7] - g[9]) * (1.f / 3.f);
  G[0] = t + g[4], G[1] = 0.5f * (g[5] - g[3]), G[2] = 0.5f * (g[6] + g[2]);
  G[3] = 0.5f * (g[5] + g[3]), G[4] = t + g[7], G[5] = 0.5f * (g[8] - g[1]);
  G[6] = 0.5f * (g[6] - g[2]), G[7] = 0.5f * (g[8] + g[1]), G[8] = t + g[9];
}
// c = a b ; c = a^T b ; c = a b^T   (3x3 row-major)
__device__ __forceinline__ void mm(const float* a, const float* b, float* c) {
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int j = 0; j < 3; j++) c[3 * i + j] = a[3 * i] * b[j] + a[3 * i + 1] * b[3 + j] + a[3 * i + 2] * b[6 + j];
}
__device__ __forceinline__ void mm_tn(const float* a, const float* b, float* c) {
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int j = 0; j < 3; j++) c[3 * i + j] = a[i] * b[j] + a[3 + i] * b[3 + j] + a[6 + i] * b[6 + j];
}
__device__ __forceinline__ void mm_nt(const float* a, const float* b, float* c) {
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int j = 0; j < 3; j++)
      c[3 * i + j] = a[3 * i] * b[3 * j] + a[3 * i + 1] * b[3 * j + 1] + a[3 * i + 2] * b[3 * j + 2];
}
__device__ __forceinline__ float norm10(const float* t) {
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < 10; k++) s = fmaf(nw_of(k) * t[k], t[k], s);
  return s;
}
__device__ __forceinline__ void load10(const float* p, int c, float* t) {
#pragma unroll
  for (int k = 0; k < 10; k++) t[k] = p[k * TC + c];
}
__device__ __forceinline__ void store10(float* p, int c, const float* t) {
#pragma unroll
  for (int k = 0; k < 10; k++) p[k * TC + c] = t[k];
}
// g_in of  out = t / (norm(t) + 1)
__device__ __forceinline__ void scale_bwd10(const float* t, float q, const float* gout, float* gin) {
  float dot = 0.f;
#pragma unroll
  for (int k = 0; k < 10; k++) dot = fmaf(gout[k], t[k], dot);
  const float rq = 1.f / q, s = dot * rq * rq;
#pragma unroll
  for (int k = 0; k < 10; k++) gin[k] = gout[k] * rq - s * 2.f * nw_of(k) * t[k];
}

#define TN_LAUNCH(kern, nitems, st, ...)                                   \
  do {                                                                     \
    if ((nitems) > 0) {                                                    \
      kern<<<cdiv((nitems), 256), 256, 0, st>>>(__VA_ARGS__);              \
      B2M_CK(cudaGetLastError());                                          \
      g_launch_count++;                                                    \
    }                                                                      \
  } while (0)

// ============================================================================================
// row GEMM  C[z][M,N] = epi(A[z][M,K] @ B[sel(z)][K,N] + bias)      (FP32 FFMA, 128x64 tile, 8x4 per thread)
// ============================================================================================
__global__ void __launch_bounds__(256) k_tn_gemm(TnGemm g) {
  __shared__ __align__(16) float As[128][36];
  __shared__ __align__(16) float Bs[32][64];
  const int tid = threadIdx.x, z = blockIdx.z;
  const int m0 = blockIdx.x * 128, n0 = blockIdx.y * 64;
  const int rg = tid >> 4, cg = tid & 15;
  const float* __restrict__ A = g.A + (size_t)z * g.zA;
  const float* __restrict__ B = g.bsel ? (z == 0 ? g.B0 : (z < 4 ? g.B1 : g.B2)) : g.B0;
  float acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; i++)
#pragma unroll
    for (int j = 0; j < 4; j++) acc[i][j] = 0.f;
  for (int k0 = 0; k0 < g.K; k0 += 32) {
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int idx = tid + 256 * i;
      const int row = idx >> 3, c4 = idx & 7;
      const int gm = m0 + row;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (gm < g.M) v = *reinterpret_cast<const float4*>(&A[(size_t)gm * g.lda + k0 + c4 * 4]);
      *reinterpret_cast<float4*>(&As[row][c4 * 4]) = v;
    }
#pragma unroll
    for (int i = 0; i < 2; i++) {
      const int idx = tid + 256 * i;
      const int kr = idx >> 4, c4 = idx & 15;
      *reinterpret_cast<float4*>(&Bs[kr][c4 * 4]) =
          *reinterpret_cast<const float4*>(&B[(size_t)(k0 + kr) * g.N + n0 + c4 * 4]);
    }
    __syncthreads();
#pragma unroll 8
    for (int k = 0; k < 32; k++) {
      const float4 b = *reinterpret_cast<const float4*>(&Bs[k][cg * 4]);
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const float a = As[rg + 16 * i][k];
        acc[i][0] = fmaf(a, b.x, acc[i][0]);
        acc[i][1] = fmaf(a, b.y, acc[i][1]);
        acc[i][2] = fmaf(a, b.z, acc[i][2]);
        acc[i][3] = fmaf(a, b.w, acc[i][3]);
      }
    }
    __syncthreads();
  }
  const int col = n0 + cg * 4;
  float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
  if (g.bias) bv = *reinterpret_cast<const float4*>(&g.bias[col]);
  float* __restrict__ C = g.C + (size_t)z * g.zC;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const int gm = m0 + rg + 16 * i;
    if (gm >= g.M) continue;
    float4 v = make_float4(acc[i][0] + bv.x, acc[i][1] + bv.y, acc[i][2] + bv.z, acc[i][3] + bv.w);
    float4* cp = reinterpret_cast<float4*>(&C[(size_t)gm * g.ldc + col]);
    if (g.epi == 1) {  // keep the pre-activation, write SiLU
      *reinterpret_cast<float4*>(&g.Cpre[(size_t)gm * g.ldc + col]) = v;
      v = make_float4(silu_f(v.x), silu_f(v.y), silu_f(v.z), silu_f(v.w));
    } else if (g.epi == 2) {  // reverse pass: times SiLU'(pre) of the layer below
      const float4 p = *reinterpret_cast<const float4*>(&g.Pre[(size_t)gm * g.ldp + col]);
      v.x *= dsilu_f(p.x), v.y *= dsilu_f(p.y), v.z *= dsilu_f(p.z), v.w *= dsilu_f(p.w);
    }
    if (g.accum) {
      const float4 c = *cp;
      v.x += c.x, v.y += c.y, v.z += c.z, v.w += c.w;
    }
    *cp = v;
  }
}

// ============================================================================================
// geometry: Gaussian expansion and cosine cutoff per edge
// ============================================================================================
__global__ void k_tn_edge_geom(int64_t E, const float4* __restrict__ e_vec, TnRadial rp, float* __restrict__ rbf,
                               float* __restrict__ cut) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= E * rp.nrp) return;
  const int64_t e = i / rp.nrp;
  const int k = (int)(i % rp.nrp);
  const float d = e_vec[e].w;
  float v = 0.f;
  if (k < rp.nr) {
    const float t = d - rp.mu[k];
    v = __expf(-rp.width * t * t);
  }
  rbf[i] = v;
  if (k == 0) cut[e] = d <= rp.rc ? 0.5f * (__cosf(CUDART_PI_F * d / rp.rc) + 1.f) : 0.f;
}

// ============================================================================================
// embedding: per destination atom, sum over incoming edges of  C(d) Z_ij (p1 I | p2 skew(v) | p3 sym(v))
// ============================================================================================
__global__ void k_tn_embed_agg(int n_own, const int* __restrict__ row_ptr, const int* __restrict__ e_src,
                               const int* __restrict__ type, const float* __restrict__ U, const float* __restrict__ V,
                               const float* __restrict__ P, const float* __restrict__ cut,
                               const float4* __restrict__ e_vec, float* __restrict__ T0, float* __restrict__ nr0) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)n_own * TC) return;
  const int t = (int)(i / TC), c = (int)(i % TC);
  float acc[10];
#pragma unroll
  for (int k = 0; k < 10; k++) acc[k] = 0.f;
  const float vt = V[(size_t)type[t] * TC + c];
  for (int e = row_ptr[t]; e < row_ptr[t + 1]; e++) {
    const float4 v = e_vec[e];
    const float rd = 1.f / v.w;
    const float x = v.x * rd, y = v.y * rd, z = v.z * rd;
    const float n3 = (x * x + y * y + z * z) * (1.f / 3.f);
    const float cz = cut[e] * (U[(size_t)type[e_src[e]] * TC + c] + vt);
    const float* p = P + (size_t)e * (3 * TC);
    const float w1 = p[c] * cz, w2 = p[TC + c] * cz, w3 = p[2 * TC + c] * cz;
    acc[0] += w1;
    acc[1] = fmaf(w2, x, acc[1]), acc[2] = fmaf(w2, y, acc[2]), acc[3] = fmaf(w2, z, acc[3]);
    acc[4] = fmaf(w3, x * x - n3, acc[4]), acc[5] = fmaf(w3, x * y, acc[5]), acc[6] = fmaf(w3, x * z, acc[6]);
    acc[7] = fmaf(w3, y * y - n3, acc[7]), acc[8] = fmaf(w3, y * z, acc[8]), acc[9] = fmaf(w3, z * z - n3, acc[9]);
  }
  store10(T0 + (size_t)t * TW, c, acc);
  nr0[(size_t)t * TC + c] = norm10(acc);
}

// LayerNorm over rows of width W (one warp per row); stats = (mean, rstd)
__global__ void k_tn_layernorm(int rows, int W, const float* __restrict__ x, const float* __restrict__ gamma,
                               const float* __restrict__ beta, float* __restrict__ y, float* __restrict__ stats) {
  const int r = (int)((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float* xr = x + (size_t)r * W;
  float s = 0.f;
  for (int c = lane; c < W; c += 32) s += xr[c];
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mu = s / (float)W;
  float v = 0.f;
  for (int c = lane; c < W; c += 32) {
    const float t = xr[c] - mu;
    v = fmaf(t, t, v);
  }
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const float rstd = rsqrtf(v / (float)W + 1e-5f);
  for (int c = lane; c < W; c += 32) y[(size_t)r * W + c] = (xr[c] - mu) * rstd * gamma[c] + beta[c];
  if (lane == 0) stats[2 * r] = mu, stats[2 * r + 1] = rstd;
}
__global__ void k_tn_layernorm_bwd(int rows, int W, const float* __restrict__ x, const float* __restrict__ stats,
                                   const float* __restrict__ gamma, const float* __restrict__ gy,
                                   float* __restrict__ gx) {
  const int r = (int)((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float mu = stats[2 * r], rstd = stats[2 * r + 1];
  const float* xr = x + (size_t)r * W;
  const float* gr = gy + (size_t)r * W;
  float s1 = 0.f, s2 = 0.f;
  for (int c = lane; c < W; c += 32) {
    const float gh = gr[c] * gamma[c], xh = (xr[c] - mu) * rstd;
    s1 += gh, s2 = fmaf(gh, xh, s2);
  }
  for (int o = 16; o > 0; o >>= 1) {
    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    s2 += __shfl_xor_sync(0xffffffffu, s2, o);
  }
  s1 /= (float)W, s2 /= (float)W;
  for (int c = lane; c < W; c += 32) {
    const float gh = gr[c] * gamma[c], xh = (xr[c] - mu) * rstd;
    gx[(size_t)r * W + c] = rstd * (gh - s1 - xh * s2);
  }
}

// X0_k = T0m_k * silu(s2p)[c, part(k)]
__global__ void k_tn_embed_out(int n, const float* __restrict__ T0m, const float* __restrict__ s2p,
                               float* __restrict__ X0) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)n * TC) return;
  const int t = (int)(i / TC), c = (int)(i % TC);
  float sc[3];
#pragma unroll
  for (int p = 0; p < 3; p++) sc[p] = silu_f(s2p[(size_t)t * (3 * TC) + 3 * c + p]);
  float v[10];
  load10(T0m + (size_t)t * TW, c, v);
#pragma unroll
  for (int k = 0; k < 10; k++) v[k] *= sc[part_of(k)];
  store10(X0 + (size_t)t * TW, c, v);
}
// gT0m_k = gX0_k * sc[part(k)] ;  gs2p[c,p] = silu'(s2p) * sum_{k in p} gX0_k T0m_k
__global__ void k_tn_embed_out_bwd(int n, const float* __restrict__ T0m, const float* __restrict__ s2p,
                                   const float* __restrict__ gX0, float* __restrict__ gT0m,
                                   float* __restrict__ gs2p) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)n * TC) return;
  const int t = (int)(i / TC), c = (int)(i % TC);
  float v[10], g[10], gs[3] = {0.f, 0.f, 0.f};
  load10(T0m + (size_t)t * TW, c, v);
  load10(gX0 + (size_t)t * TW, c, g);
#pragma unroll
  for (int k = 0; k < 10; k++) gs[part_of(k)] = fmaf(g[k], v[k], gs[part_of(k)]);
#pragma unroll
  for (int p = 0; p < 3; p++) {
    const float pre = s2p[(size_t)t * (3 * TC) + 3 * c + p];
    gs2p[(size_t)t * (3 * TC) + 3 * c + p] = gs[p] * dsilu_f(pre);
    gs[p] = silu_f(pre);
  }
#pragma unroll
  for (int k = 0; k < 10; k++) g[k] *= gs[part_of(k)];
  store10(gT0m + (size_t)t * TW, c, g);
}
// gT0_k += gnr0 * 2 nw_k T0_k
__global__ void k_tn_norm_bwd_add(int n, const float* __restrict__ T0, const float* __restrict__ gnr0,
                                  float* __restrict__ gT0) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)n * TC) return;
  const int t = (int)(i / TC), c = (int)(i % TC);
  const float gn = gnr0[(size_t)t * TC + c];
#pragma unroll
  for (int k = 0; k < 10; k++) {
    const size_t o = (size_t)t * TW + k * TC + c;
    gT0[o] = fmaf(gn * 2.f * nw_of(k), T0[o], gT0[o]);
  }
}

// reverse of k_tn_embed_agg, one warp per edge (lanes own channels lane and lane + 32):
//   gP[e] (3C), gC[e] += , gvh[e] (3)
__global__ void k_tn_embed_agg_bwd(int64_t E, const int* __restrict__ e_src, const int* __restrict__ e_dst,
                                   const int* __restrict__ type, const float* __restrict__ U,
                                   const float* __restrict__ V, const float* __restrict__ P,
                                   const float* __restrict__ cut, const float4* __restrict__ e_vec,
                                   const float* __restrict__ gT0, float* __restrict__ gP, float* __restrict__ gC,
                                   float* __restrict__ gvh) {
  const int64_t e = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (e >= E) return;
  const int s = e_src[e], t = e_dst[e];
  const float4 v = e_vec[e];
  const float rd = 1.f / v.w;
  const float x = v.x * rd, y = v.y * rd, z = v.z * rd;
  const float n3 = (x * x + y * y + z * z) * (1.f / 3.f);
  const float s6[6] = {x * x - n3, x * y, x * z, y * y - n3, y * z, z * z - n3};
  const float ce = cut[e];
  float rC = 0.f, a3[3] = {0.f, 0.f, 0.f}, w6[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int h = 0; h < 2; h++) {
    const int c = lane + 32 * h;
    const float zij = U[(size_t)type[s] * TC + c] + V[(size_t)type[t] * TC + c];
    const float cz = ce * zij;
    float g[10];
    load10(gT0 + (size_t)t * TW, c, g);
    const float* p = P + (size_t)e * (3 * TC);
    const float p1 = p[c], p2 = p[TC + c], p3 = p[2 * TC + c];
    const float dA = g[1] * x + g[2] * y + g[3] * z;
    float dS = 0.f;
#pragma unroll
    for (int q = 0; q < 6; q++) dS = fmaf(g[4 + q], s6[q], dS);
    float* gp = gP + (size_t)e * (3 * TC);
    gp[c] = g[0] * cz, gp[TC + c] = dA * cz, gp[2 * TC + c] = dS * cz;
    rC += zij * (g[0] * p1 + p2 * dA + p3 * dS);
#pragma unroll
    for (int a = 0; a < 3; a++) a3[a] = fmaf(g[1 + a] * cz, p2, a3[a]);
#pragma unroll
    for (int q = 0; q < 6; q++) w6[q] = fmaf(g[4 + q] * cz, p3, w6[q]);
  }
  for (int o = 16; o > 0; o >>= 1) {
    rC += __shfl_xor_sync(0xffffffffu, rC, o);
#pragma unroll
    for (int a = 0; a < 3; a++) a3[a] += __shfl_xor_sync(0xffffffffu, a3[a], o);
#pragma unroll
    for (int q = 0; q < 6; q++) w6[q] += __shfl_xor_sync(0xffffffffu, w6[q], o);
  }
  if (lane == 0) {
    const float tr = w6[0] + w6[3] + w6[5];
    gC[e] += rC;
    gvh[3 * e] = a3[0] + 2.f * w6[0] * x + w6[1] * y + w6[2] * z - (2.f / 3.f) * x * tr;
    gvh[3 * e + 1] = a3[1] + w6[1] * x + 2.f * w6[3] * y + w6[4] * z - (2.f / 3.f) * y * tr;
    gvh[3 * e + 2] = a3[2] + w6[2] * x + w6[4] * y + 2.f * w6[5] * z - (2.f / 3.f) * z * tr;
  }
}

// ============================================================================================
// interaction layer, node side
// ============================================================================================
// Xh = X / (norm(X) + 1)
__global__ void k_tn_scale(int n, const float* __restrict__ X, float* __restrict__ Xh, float* __restrict__ q) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)n * TC) return;
  const int t = (int)(i / TC), c = (int)(i % TC);
  float v[10];
  load10(X + (size_t)t * TW, c, v);
  const float qq = norm10(v) + 1.f, rq = 1.f / qq;
#pragma unroll
  for (int k = 0; k < 10; k++) v[k] *= rq;
  store10(Xh + (size_t)t * TW, c, v);
  q[(size_t)t * TC + c] = qq;
}
// in place: g <- adjoint of X given adjoint of Xh
__global__ void k_tn_scale_bwd(int n, const float* __restrict__ X, const float* __restrict__ q, float* __restrict__ g) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)n * TC) return;
  const int t = (int)(i / TC), c = (int)(i % TC);
  float v[10], go[10], gi[10];
  load10(X + (size_t)t * TW, c, v);
  load10(g + (size_t)t * TW, c, go);
  scale_bwd10(v, q[(size_t)t * TC + c], go, gi);
  store10(g + (size_t)t * TW, c, gi);
}

// msg[t] = sum_{e -> t} silu(f3p[e])[c, part] C(d_e) * Y[src(e)]
__global__ void k_tn_msg(int n_own, const int* __restrict__ row_ptr, const int* __restrict__ e_src,
                         const float* __restrict__ f3p, const float* __restrict__ cut, const float* __restrict__ Y,
                         float* __restrict__ msg) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)n_own * TC) return;
  const int t = (int)(i / TC), c = (int)(i % TC);
  float acc[10];
#pragma unroll
  for (int k = 0; k < 10; k++) acc[k] = 0.f;
  for (int e = row_ptr[t]; e < row_ptr[t + 1]; e++) {
    const float ce = cut[e];
    const float* fp = f3p + (size_t)e * (3 * TC) + 3 * c;
    const float f[3] = {silu_f(fp[0]) * ce, silu_f(fp[1]) * ce, silu_f(fp[2]) * ce};
    const float* ys = Y + (size_t)e_src[e] * TW;
#pragma unroll
    for (int k = 0; k < 10; k++) acc[k] = fmaf(f[part_of(k)], ys[k * TC + c], acc[k]);
  }
  store10(msg + (size_t)t * TW, c, acc);
}
// reverse of k_tn_msg with the activation folded in (fe = silu(f3p) C):
//   g3[e][c,p] = C silu'(f3p) sum_{k in p} gmsg[t]_k Y[s]_k      (adjoint of the edge MLP's last pre-activation)
//   gC[e]     += sum_{c,p} silu(f3p) (...)                        (one warp = 32 channels of one destination: shuffle sum)
//   gY[s]_k   += fe[e][c,part(k)] gmsg[t]_k
__global__ void k_tn_msg_bwd(int n_own, const int* __restrict__ row_ptr, const int* __restrict__ e_src,
                             const float* __restrict__ f3p, const float* __restrict__ cut,
                             const float* __restrict__ Y, const float* __restrict__ gmsg, float* __restrict__ g3,
                             float* __restrict__ gC, float* __restrict__ gY) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)n_own * TC) return;  // n_own * 64 is a multiple of 32: whole warps leave together
  const int t = (int)(i / TC), c = (int)(i % TC), lane = threadIdx.x & 31;
  float gm[10];
  load10(gmsg + (size_t)t * TW, c, gm);
  for (int e = row_ptr[t]; e < row_ptr[t + 1]; e++) {
    const float ce = cut[e];
    const float* fp = f3p + (size_t)e * (3 * TC) + 3 * c;
    const float pre[3] = {fp[0], fp[1], fp[2]};
    float sl[3], f[3];
#pragma unroll
    for (int p = 0; p < 3; p++) sl[p] = silu_f(pre[p]), f[p] = sl[p] * ce;
    const size_t so = (size_t)e_src[e] * TW;
    float gq[3] = {0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < 10; k++) {
      gq[part_of(k)] = fmaf(gm[k], Y[so + k * TC + c], gq[part_of(k)]);
      atomicAdd(&gY[so + k * TC + c], f[part_of(k)] * gm[k]);
    }
    float* go = g3 + (size_t)e * (3 * TC) + 3 * c;
    float sc = 0.f;
#pragma unroll
    for (int p = 0; p < 3; p++) {
      go[p] = gq[p] * ce * dsilu_f(pre[p]);
      sc = fmaf(gq[p], sl[p], sc);
    }
    for (int o = 16; o > 0; o >>= 1) sc += __shfl_xor_sync(0xffffffffu, sc, o);
    if (lane == 0) atomicAdd(&gC[e], sc);
  }
}

// Pn = dec(P) / (norm + 1),  P = msg Y + Y msg  (O(3))  |  2 Y msg  (SO(3))
__device__ __forceinline__ void tn_product(const float* m10, const float* y10, int so3, float* pd) {
  float M[9], Yf[9], A[9], B[9];
  full9(m10, M), full9(y10, Yf);
  mm(Yf, M, B);
  if (so3) {
#pragma unroll
    for (int k = 0; k < 9; k++) A[k] = 2.f * B[k];
  } else {
    mm(M, Yf, A);
#pragma unroll
    for (int k = 0; k < 9; k++) A[k] += B[k];
  }
  dec10(A, pd);
}
__global__ void k_tn_prod(int n, const float* __restrict__ msg, const float* __restrict__ Y, int so3,
                          float* __restrict__ Pn) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)n * TC) return;
  const int t = (int)(i / TC), c = (int)(i % TC);
  float m[10], y[10], pd[10];
  load10(msg + (size_t)t * TW, c, m);
  load10(Y + (size_t)t * TW, c, y);
  tn_product(m, y, so3, pd);
  const float rq = 1.f / (norm10(pd) + 1.f);
#pragma unroll
  for (int k = 0; k < 10; k++) pd[k] *= rq;
  store10(Pn + (size_t)t * TW, c, pd);
}
// gPn -> gmsg (set), gY (set, owned rows)
__global__ void k_tn_prod_bwd(int n, const float* __restrict__ msg, const float* __restrict__ Y, int so3,
                              const float* __restrict__ gPn, float* __restrict__ gmsg, float* __restrict__ gY) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)n * TC) return;
  const int t = (int)(i / TC), c = (int)(i % TC);
  float m[10], y[10], pd[10], go[10], gpd[10];
  load10(msg + (size_t)t * TW, c, m);
  load10(Y + (size_t)t * TW, c, y);
  load10(gPn + (size_t)t * TW, c, go);
  tn_product(m, y, so3, pd);
  scale_bwd10(pd, norm10(pd) + 1.f, go, gpd);
  float G[9], M[9], Yf[9], gM[9], gYf[9], T1[9];
  dec_adj(gpd, G);
  full9(m, M), full9(y, Yf);
  if (so3) {  // P = 2 Y M : gM = 2 Y^T G, gY = 2 G M^T
    mm_tn(Yf, G, gM), mm_nt(G, M, gYf);
#pragma unroll
    for (int k = 0; k < 9; k++) gM[k] *= 2.f, gYf[k] *= 2.f;
  } else {  // P = M Y + Y M : gM = G Y^T + Y^T G, gY = M^T G + G M^T
    mm_nt(G, Yf, gM), mm_tn(Yf, G, T1);
#pragma unroll
    for (int k = 0; k < 9; k++) gM[k] += T1[k];
    mm_tn(M, G, gYf), mm_nt(G, M, T1);
#pragma unroll
    for (int k = 0; k < 9; k++) gYf[k] += T1[k];
  }
  full_adj(gM, go), full_adj(gYf, gpd);
  store10(gmsg + (size_t)t * TW, c, go);
  store10(gY + (size_t)t * TW, c, gpd);
}

// Xn = Xh + dX + dec(full(dX)^2)
__global__ void k_tn_update(int n, const float* __restrict__ Xh, const float* __restrict__ dX, float* __restrict__ Xn) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)n * TC) return;
  const int t = (int)(i / TC), c = (int)(i % TC);
  float xh[10], d[10], Df[9], D2[9], sq[10];
  load10(Xh + (size_t)t * TW, c, xh);
  load10(dX + (size_t)t * TW, c, d);
  full9(d, Df);
  mm(Df, Df, D2);
  dec10(D2, sq);
#pragma unroll
  for (int k = 0; k < 10; k++) xh[k] += d[k] + sq[k];
  store10(Xn + (size_t)t * TW, c, xh);
}
// gdX = gXn + full_adj(G D^T + D^T G), G = dec_adj(gXn)      (gXh = gXn: the caller reuses the buffer)
__global__ void k_tn_update_bwd(int n, const float* __restrict__ dX, const float* __restrict__ gXn,
                                float* __restrict__ gdX) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)n * TC) return;
  const int t = (int)(i / TC), c = (int)(i % TC);
  float d[10], g[10], Df[9], G[9], T1[9], T2[9], ga[10];
  load10(dX + (size_t)t * TW, c, d);
  load10(gXn + (size_t)t * TW, c, g);
  full9(d, Df);
  dec_adj(g, G);
  mm_nt(G, Df, T1), mm_tn(Df, G, T2);
#pragma unroll
  for (int k = 0; k < 9; k++) T1[k] += T2[k];
  full_adj(T1, ga);
#pragma unroll
  for (int k = 0; k < 10; k++) g[k] += ga[k];
  store10(gdX + (size_t)t * TW, c, g);
}

// ============================================================================================
// readout
// ============================================================================================
// inv = [ |I|^2 , |A|^2 , |S|^2 ]  (3C per atom)
__global__ void k_tn_invariants(int n, const float* __restrict__ X, float* __restrict__ inv) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)n * TC) return;
  const int t = (int)(i / TC), c = (int)(i % TC);
  float v[10], s[3] = {0.f, 0.f, 0.f};
  load10(X + (size_t)t * TW, c, v);
#pragma unroll
  for (int k = 0; k < 10; k++) s[part_of(k)] = fmaf(nw_of(k) * v[k], v[k], s[part_of(k)]);
#pragma unroll
  for (int p = 0; p < 3; p++) inv[(size_t)t * (3 * TC) + p * TC + c] = s[p];
}
__global__ void k_tn_invariants_bwd(int n, const float* __restrict__ X, const float* __restrict__ ginv,
                                    float* __restrict__ gX) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)n * TC) return;
  const int t = (int)(i / TC), c = (int)(i % TC);
  float v[10];
  load10(X + (size_t)t * TW, c, v);
#pragma unroll
  for (int k = 0; k < 10; k++) v[k] *= 2.f * nw_of(k) * ginv[(size_t)t * (3 * TC) + part_of(k) * TC + c];
  store10(gX + (size_t)t * TW, c, v);
}
// last layer of both readout chains (width W -> 1), product, energy sum; one warp per atom
__global__ void k_tn_readout_final(int n, int W, const float* __restrict__ hL, const float* __restrict__ wL, float bL,
                                   const float* __restrict__ hG, const float* __restrict__ wG, float bG,
                                   const int* __restrict__ type, const double* __restrict__ eref, float scale,
                                   float* __restrict__ lout, float* __restrict__ gout, float* __restrict__ e_atom,
                                   double* __restrict__ energy) {
  const int r = (int)((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (r >= n) return;
  float a = 0.f, b = 0.f;
  for (int c = lane; c < W; c += 32) {
    a = fmaf(hL[(size_t)r * W + c], wL[c], a);
    b = fmaf(hG[(size_t)r * W + c], wG[c], b);
  }
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o);
    b += __shfl_xor_sync(0xffffffffu, b, o);
  }
  if (lane == 0) {
    const float L = a + bL, Gt = sigm(b + bG);
    lout[r] = L, gout[r] = Gt, e_atom[r] = L * Gt;
    double ev = (double)scale * (double)(L * Gt);
    if (eref) ev += eref[type[r]];
    atomicAdd(energy, ev);
  }
}
// adjoints of the last hidden activations of both chains, already times SiLU'(pre) of that layer
__global__ void k_tn_readout_seed(int n, int W, const float* __restrict__ lout, const float* __restrict__ gout,
                                  float scale, const float* __restrict__ wL, const float* __restrict__ wG,
                                  const float* __restrict__ preL, const float* __restrict__ preG,
                                  float* __restrict__ gL, float* __restrict__ gG) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)n * W) return;
  const int r = (int)(i / W), c = (int)(i % W);
  const float L = lout[r], Gt = gout[r];
  gL[i] = scale * Gt * wL[c] * dsilu_f(preL[i]);
  gG[i] = scale * L * Gt * (1.f - Gt) * wG[c] * dsilu_f(preG[i]);
}

// ============================================================================================
// final geometry reverse: gd = g_rbf . drbf/dd + gC C'(d);  g_vec = gd v^ + (gvh - (gvh.v^) v^) / d
// ============================================================================================
__device__ __forceinline__ void virial_reduce_tn(const float (&v)[9], double* __restrict__ virial) {
  __shared__ float red[9][8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int k = 0; k < 9; k++) {
    float x = v[k];
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if (lane == 0) red[k][warp] = x;
  }
  __syncthreads();
  if (threadIdx.x < 9) {
    double s = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) s += (double)red[threadIdx.x][w];
    atomicAdd(&virial[threadIdx.x], s);
  }
}
// kPerAtom: also W_i (peratom.cuh) into atom_vir; the false instance is the plain kernel (atom_vir unused)
template <bool kPerAtom>
__global__ void __launch_bounds__(256) k_tn_edge_final(int64_t E, const int* __restrict__ e_src,
                                                       const int* __restrict__ e_dst, const float4* __restrict__ e_vec,
                                                       const int* __restrict__ gid, TnRadial rp,
                                                       const float* __restrict__ g_rbf, const float* __restrict__ gC,
                                                       const float* __restrict__ gvh, float* __restrict__ gd_out,
                                                       float* __restrict__ forces, double* __restrict__ virial,
                                                       float* __restrict__ atom_vir) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  float vir[9];
#pragma unroll
  for (int k = 0; k < 9; k++) vir[k] = 0.f;
  int pa_dst = -1, pa_src = 0;
  if (e < E) {
    const float4 v = e_vec[e];
    const float d = v.w, rd = 1.f / d;
    float gd = 0.f;
    for (int k = 0; k < rp.nr; k++) {
      const float t = d - rp.mu[k];
      gd = fmaf(g_rbf[(size_t)e * rp.nrp + k], __expf(-rp.width * t * t) * (-2.f * rp.width * t), gd);
    }
    if (d <= rp.rc) gd = fmaf(gC[e], -0.5f * CUDART_PI_F / rp.rc * __sinf(CUDART_PI_F * d / rp.rc), gd);
    gd_out[e] = gd;
    const float x = v.x * rd, y = v.y * rd, z = v.z * rd;
    const float hx = gvh[3 * e], hy = gvh[3 * e + 1], hz = gvh[3 * e + 2];
    const float pr = hx * x + hy * y + hz * z;
    const float gx = gd * x + (hx - pr * x) * rd, gy = gd * y + (hy - pr * y) * rd, gz = gd * z + (hz - pr * z) * rd;
    // vec = x_dst + off.L - x_src :  dE/dx_dst += g, dE/dx_src -= g ; F = -dE/dx   (pes.py:122-124)
    const int gdst = gid[e_dst[e]], gsrc = gid[e_src[e]];
    if constexpr (kPerAtom) pa_dst = gdst, pa_src = gsrc;
    atomicAdd(&forces[(size_t)gdst * 3], -gx);
    atomicAdd(&forces[(size_t)gdst * 3 + 1], -gy);
    atomicAdd(&forces[(size_t)gdst * 3 + 2], -gz);
    atomicAdd(&forces[(size_t)gsrc * 3], gx);
    atomicAdd(&forces[(size_t)gsrc * 3 + 1], gy);
    atomicAdd(&forces[(size_t)gsrc * 3 + 2], gz);
    vir[0] = v.x * gx, vir[1] = v.x * gy, vir[2] = v.x * gz;  // strain_bar[a][b] = sum vec[a] g[b]  (pes.py:140-145)
    vir[3] = v.y * gx, vir[4] = v.y * gy, vir[5] = v.y * gz;
    vir[6] = v.z * gx, vir[7] = v.z * gy, vir[8] = v.z * gz;
  }
  if constexpr (kPerAtom) atom_vir_edge(atom_vir, pa_dst, pa_src, vir);
  virial_reduce_tn(vir, virial);
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------
void launch_tn_gemm(cudaStream_t st, const TnGemm& g, int nz) {
  if (g.M <= 0) return;
  B2M_REQUIRE(g.K % 32 == 0 && g.N % 64 == 0 && g.lda % 4 == 0 && g.ldc % 4 == 0, B2M_ERR_INVALID, "tn gemm shape");
  B2M_REQUIRE(g.epi == 0 || (nz == 1 && (g.epi == 1 ? g.Cpre != nullptr : g.Pre != nullptr)), B2M_ERR_INVALID,
              "tn gemm epilogue");  // the epilogue pointers carry no z offset
  dim3 grid(cdiv(g.M, 128), g.N / 64, nz);
  k_tn_gemm<<<grid, 256, 0, st>>>(g);
  B2M_CK(cudaGetLastError());
  g_launch_count++;
}
void launch_tn_edge_geom(cudaStream_t st, int64_t E, const float4* e_vec, const TnRadial& rp, float* rbf, float* cut) {
  TN_LAUNCH(k_tn_edge_geom, E * rp.nrp, st, E, e_vec, rp, rbf, cut);
}
void launch_tn_embed_agg(cudaStream_t st, int n_own, const int* row_ptr, const int* e_src, const int* type,
                         const float* U, const float* V, const float* P, const float* cut, const float4* e_vec,
                         float* T0, float* nr0) {
  TN_LAUNCH(k_tn_embed_agg, (int64_t)n_own * TC, st, n_own, row_ptr, e_src, type, U, V, P, cut, e_vec, T0, nr0);
}
void launch_tn_layernorm(cudaStream_t st, int rows, int W, const float* x, const float* gamma, const float* beta,
                         float* y, float* stats) {
  TN_LAUNCH(k_tn_layernorm, (int64_t)rows * 32, st, rows, W, x, gamma, beta, y, stats);
}
void launch_tn_layernorm_bwd(cudaStream_t st, int rows, int W, const float* x, const float* stats, const float* gamma,
                             const float* gy, float* gx) {
  TN_LAUNCH(k_tn_layernorm_bwd, (int64_t)rows * 32, st, rows, W, x, stats, gamma, gy, gx);
}
void launch_tn_embed_out(cudaStream_t st, int n, const float* T0m, const float* s2p, float* X0) {
  TN_LAUNCH(k_tn_embed_out, (int64_t)n * TC, st, n, T0m, s2p, X0);
}
void launch_tn_embed_out_bwd(cudaStream_t st, int n, const float* T0m, const float* s2p, const float* gX0, float* gT0m,
                             float* gs2p) {
  TN_LAUNCH(k_tn_embed_out_bwd, (int64_t)n * TC, st, n, T0m, s2p, gX0, gT0m, gs2p);
}
void launch_tn_norm_bwd_add(cudaStream_t st, int n, const float* T0, const float* gnr0, float* gT0) {
  TN_LAUNCH(k_tn_norm_bwd_add, (int64_t)n * TC, st, n, T0, gnr0, gT0);
}
void launch_tn_embed_agg_bwd(cudaStream_t st, int64_t E, const int* e_src, const int* e_dst, const int* type,
                             const float* U, const float* V, const float* P, const float* cut, const float4* e_vec,
                             const float* gT0, float* gP, float* gC, float* gvh) {
  TN_LAUNCH(k_tn_embed_agg_bwd, E * 32, st, E, e_src, e_dst, type, U, V, P, cut, e_vec, gT0, gP, gC, gvh);
}
void launch_tn_scale(cudaStream_t st, int n, const float* X, float* Xh, float* q) {
  TN_LAUNCH(k_tn_scale, (int64_t)n * TC, st, n, X, Xh, q);
}
void launch_tn_scale_bwd(cudaStream_t st, int n, const float* X, const float* q, float* g) {
  TN_LAUNCH(k_tn_scale_bwd, (int64_t)n * TC, st, n, X, q, g);
}
void launch_tn_msg(cudaStream_t st, int n_own, const int* row_ptr, const int* e_src, const float* f3p, const float* cut,
                   const float* Y, float* msg) {
  TN_LAUNCH(k_tn_msg, (int64_t)n_own * TC, st, n_own, row_ptr, e_src, f3p, cut, Y, msg);
}
void launch_tn_msg_bwd(cudaStream_t st, int n_own, const int* row_ptr, const int* e_src, const float* f3p,
                       const float* cut, const float* Y, const float* gmsg, float* g3, float* gC, float* gY) {
  TN_LAUNCH(k_tn_msg_bwd, (int64_t)n_own * TC, st, n_own, row_ptr, e_src, f3p, cut, Y, gmsg, g3, gC, gY);
}
void launch_tn_prod(cudaStream_t st, int n, const float* msg, const float* Y, int so3, float* Pn) {
  TN_LAUNCH(k_tn_prod, (int64_t)n * TC, st, n, msg, Y, so3, Pn);
}
void launch_tn_prod_bwd(cudaStream_t st, int n, const float* msg, const float* Y, int so3, const float* gPn,
                        float* gmsg, float* gY) {
  TN_LAUNCH(k_tn_prod_bwd, (int64_t)n * TC, st, n, msg, Y, so3, gPn, gmsg, gY);
}
void launch_tn_update(cudaStream_t st, int n, const float* Xh, const float* dX, float* Xn) {
  TN_LAUNCH(k_tn_update, (int64_t)n * TC, st, n, Xh, dX, Xn);
}
void launch_tn_update_bwd(cudaStream_t st, int n, const float* dX, const float* gXn, float* gdX) {
  TN_LAUNCH(k_tn_update_bwd, (int64_t)n * TC, st, n, dX, gXn, gdX);
}
void launch_tn_invariants(cudaStream_t st, int n, const float* X, float* inv) {
  TN_LAUNCH(k_tn_invariants, (int64_t)n * TC, st, n, X, inv);
}
void launch_tn_invariants_bwd(cudaStream_t st, int n, const float* X, const float* ginv, float* gX) {
  TN_LAUNCH(k_tn_invariants_bwd, (int64_t)n * TC, st, n, X, ginv, gX);
}
void launch_tn_readout_final(cudaStream_t st, int n, int W, const float* hL, const float* wL, float bL, const float* hG,
                             const float* wG, float bG, const int* type, const double* eref, float scale, float* lout,
                             float* gout, float* e_atom, double* energy) {
  TN_LAUNCH(k_tn_readout_final, (int64_t)n * 32, st, n, W, hL, wL, bL, hG, wG, bG, type, eref, scale, lout, gout,
            e_atom, energy);
}
void launch_tn_readout_seed(cudaStream_t st, int n, int W, const float* lout, const float* gout, float scale,
                            const float* wL, const float* wG, const float* preL, const float* preG, float* gL,
                            float* gG) {
  TN_LAUNCH(k_tn_readout_seed, (int64_t)n * W, st, n, W, lout, gout, scale, wL, wG, preL, preG, gL, gG);
}
void launch_tn_edge_final(cudaStream_t st, int64_t E, const int* e_src, const int* e_dst, const float4* e_vec,
                          const int* gid, const TnRadial& rp, const float* g_rbf, const float* gC, const float* gvh,
                          float* gd, float* forces, double* virial, float* atom_vir) {
  if (atom_vir)
    TN_LAUNCH(k_tn_edge_final<true>, E, st, E, e_src, e_dst, e_vec, gid, rp, g_rbf, gC, gvh, gd, forces, virial, atom_vir);
  else
    TN_LAUNCH(k_tn_edge_final<false>, E, st, E, e_src, e_dst, e_vec, gid, rp, g_rbf, gC, gvh, gd, forces, virial, nullptr);
}

}  // namespace b2m
