// kernels.cu -- hand-written sm_100a kernels of the CHGNet hot path (fp32 FFMA math,
// cp.async.bulk (TMA) row gathers into shared memory, segmented scatter-adds).
// See kernels.cuh for the formulation; oracle/manual_ref.py is the CPU mirror of every stage.
#include "kernels.cuh"
#include "peratom.cuh"

namespace b2m {

std::atomic<long long> g_launch_count{0};

// ============================================================================================
// device helpers
// ============================================================================================
// MUFU.EX2 + MUFU.RCP, flush-to-zero forms (same bits as __fdividef/__expf for normal results, no range fix-ups)
__device__ __forceinline__ float sigm(float x) {
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * -1.4426950408889634f));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.f + e));
  return r;
}
__device__ __forceinline__ float silu_f(float x) { return x * sigm(x); }
__device__ __forceinline__ float dsilu_f(float x) {
  float s = sigm(x);
  return s * (1.f + x * (1.f - s));
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// TMA bulk copy global -> shared (one row), completion signalled on an mbarrier
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok = 0;
  const uint32_t addr = smem_u32(bar);
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
  } while (!ok);
}

__device__ __forceinline__ float ipowf(float x, int n) {
  float r = 1.f;
  for (int i = 0; i < n; i++) r *= x;
  return r;
}
// be_k = env(rbf_k) rbf_k with the envelope applied to the rbf VALUE (chgnet.py:116-124), and d be_k / dd
__device__ __forceinline__ void rbf_env_k(float d, float freq, const RadialParams& rp, float& be, float& dbe) {
  const float invd = 1.f / d;
  const float w = freq / rp.rc;
  float s, c;
  sincosf(d * w, &s, &c);
  const float rbf = rp.norm * s * invd;
  const float drbf = rp.norm * (w * c * invd - s * invd * invd);
  const int p = rp.p;
  const float c1 = -(p + 1) * (p + 2) * 0.5f, c2 = (float)(p * (p + 2)), c3 = -p * (p + 1) * 0.5f;
  const float rho = rbf / rp.rc;
  const float rm1 = ipowf(rho, p - 1);
  const float r0 = rm1 * rho, r1 = r0 * rho, r2 = r1 * rho;
  const float env = 1.f + c1 * r0 + c2 * r1 + c3 * r2;
  const float denv = (c1 * p * rm1 + c2 * (p + 1) * r0 + c3 * (p + 2) * r1) / rp.rc;
  const bool ok = rbf <= rp.rc;
  be = ok ? env * rbf : 0.f;
  dbe = ok ? (env + rbf * denv) * drbf : 0.f;
}

// thread -> micro-tile mapping of the 256-thread fused kernels:
//   branch = tid>>7 (0: "layers", 1: "gates"), rows r_i = rg + 16 i, cols c_j = cg*4 + (j&3) + 32 (j>>2)
struct Map {
  int branch, rg, cg;
  __device__ __forceinline__ Map() {
    const int tid = threadIdx.x;
    branch = tid >> 7;
    const int t128 = tid & 127, lane = tid & 31;
    rg = (t128 >> 5) * 4 + (lane >> 3);
    cg = lane & 7;
  }
  __device__ __forceinline__ int row(int i) const { return rg + 16 * i; }
  __device__ __forceinline__ int col(int j) const { return cg * 4 + (j & 3) + 32 * (j >> 2); }
};

// acc[8][8] += At[r_i][kofs + k] * Wk[k][c_j], k < 64.  At: smem row-major pitch lda; Wk: smem [64][64].
__device__ __forceinline__ void gemm64(const float* __restrict__ At, int lda, int kofs, const float* __restrict__ Wk,
                                       float (&acc)[8][8], const Map& m) {
  const float* a0 = At + m.rg * lda + kofs;
  const float* w0p = Wk + m.cg * 4;
#pragma unroll 4
  for (int k = 0; k < 64; k++) {
    const float4 w0 = *reinterpret_cast<const float4*>(w0p + k * 64);
    const float4 w1 = *reinterpret_cast<const float4*>(w0p + k * 64 + 32);
#pragma unroll
    for (int i = 0; i < 8; i++) {
      const float av = a0[i * 16 * lda + k];
      acc[i][0] = fmaf(av, w0.x, acc[i][0]);
      acc[i][1] = fmaf(av, w0.y, acc[i][1]);
      acc[i][2] = fmaf(av, w0.z, acc[i][2]);
      acc[i][3] = fmaf(av, w0.w, acc[i][3]);
      acc[i][4] = fmaf(av, w1.x, acc[i][4]);
      acc[i][5] = fmaf(av, w1.y, acc[i][5]);
      acc[i][6] = fmaf(av, w1.z, acc[i][6]);
      acc[i][7] = fmaf(av, w1.w, acc[i][7]);
    }
  }
}

__device__ __forceinline__ void stage_w(float* Wsm, const float* __restrict__ g, int nfloat4) {
  for (int i = threadIdx.x; i < nfloat4; i += NT) reinterpret_cast<float4*>(Wsm)[i] = reinterpret_cast<const float4*>(g)[i];
}

// running segmented sum over rows [r0, r1) of a smem tile column, flushed with atomics when the key changes
__device__ __forceinline__ void seg_flush(const float* tile, int ld, int col, int r0, int r1, const int* key,
                                          float* __restrict__ out, int width) {
  float sum = 0.f;
  int cur = -1;
  for (int r = r0; r < r1; r++) {
    const int k = key[r];
    if (k != cur) {
      if (cur >= 0) atomicAdd(&out[(size_t)cur * width + col], sum);
      cur = k;
      sum = 0.f;
    }
    if (k >= 0) sum += tile[r * ld + col];
  }
  if (cur >= 0) atomicAdd(&out[(size_t)cur * width + col], sum);
}

// ============================================================================================
// generic row GEMM (node-level projections; ~10% of the FLOPs)
// ============================================================================================
__global__ void __launch_bounds__(256) k_gemm(const float* __restrict__ A, int lda, const float* __restrict__ B,
                                              float* __restrict__ C, int ldc, int M, int N, int K,
                                              const float* __restrict__ bias, const float* __restrict__ R, int ldr,
                                              int accum) {
  __shared__ __align__(16) float As[128][36];
  __shared__ __align__(16) float Bs[32][64];
  const int tid = threadIdx.x;
  const int m0 = blockIdx.x * 128, n0 = blockIdx.y * 64;
  const int rg = tid >> 4, cg = tid & 15;
  float acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; i++)
    for (int j = 0; j < 4; j++) acc[i][j] = 0.f;
  for (int k0 = 0; k0 < K; k0 += 32) {
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int idx = tid + 256 * i;
      const int row = idx >> 3, c4 = idx & 7;
      const int gm = m0 + row;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (gm < M) v = *reinterpret_cast<const float4*>(&A[(size_t)gm * lda + k0 + c4 * 4]);
      *reinterpret_cast<float4*>(&As[row][c4 * 4]) = v;
    }
#pragma unroll
    for (int i = 0; i < 2; i++) {
      const int idx = tid + 256 * i;
      const int kr = idx >> 4, c4 = idx & 15;
      *reinterpret_cast<float4*>(&Bs[kr][c4 * 4]) =
          *reinterpret_cast<const float4*>(&B[(size_t)(k0 + kr) * N + n0 + c4 * 4]);
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
  if (bias) bv = *reinterpret_cast<const float4*>(&bias[col]);
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const int gm = m0 + rg + 16 * i;
    if (gm >= M) continue;
    float4 v = make_float4(acc[i][0] + bv.x, acc[i][1] + bv.y, acc[i][2] + bv.z, acc[i][3] + bv.w);
    if (R) {
      const float4 r = *reinterpret_cast<const float4*>(&R[(size_t)gm * ldr + col]);
      v.x += r.x, v.y += r.y, v.z += r.z, v.w += r.w;
    }
    float4* cp = reinterpret_cast<float4*>(&C[(size_t)gm * ldc + col]);
    if (accum) {
      const float4 c = *cp;
      v.x += c.x, v.y += c.y, v.z += c.z, v.w += c.w;
    }
    *cp = v;
  }
}

void launch_gemm(cudaStream_t st, const float* A, int lda, const float* B, float* C, int ldc, int M, int N, int K,
                 const float* bias, const float* R, int ldr, bool accum) {
  if (M <= 0) return;
  B2M_REQUIRE(K % 32 == 0 && N % 64 == 0, B2M_ERR_INVALID, "gemm shape");
  dim3 grid(cdiv(M, 128), N / 64);
  k_gemm<<<grid, 256, 0, st>>>(A, lda, B, C, ldc, M, N, K, bias, R, ldr, accum ? 1 : 0);
  B2M_CK(cudaGetLastError());
  g_launch_count++;
}

// ============================================================================================
// small elementwise / init kernels
// ============================================================================================
__global__ void k_embed(int n, const int* __restrict__ type, const float* __restrict__ emb, float* __restrict__ x0) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)n * 16) return;
  const int r = (int)(i >> 4), c4 = (int)(i & 15);
  reinterpret_cast<float4*>(x0)[(size_t)r * 16 + c4] = reinterpret_cast<const float4*>(emb)[(size_t)type[r] * 16 + c4];
}
void launch_embed(cudaStream_t st, int n, const int* type, const float* emb, float* x0) {
  if (n <= 0) return;
  k_embed<<<cdiv((int64_t)n * 16, 256), 256, 0, st>>>(n, type, emb, x0);
  B2M_CK(cudaGetLastError());
  g_launch_count++;
}

// out[b][c] = sum_k be_k(d_b) W[c][k]     (32 bonds per block)
__global__ void __launch_bounds__(256) k_bond_init(int nb, const float4* __restrict__ b_vec, RadialParams rp,
                                                   const float* __restrict__ W, float* __restrict__ out) {
  __shared__ float be_s[32][12];
  __shared__ float Ws[64 * 9];
  const int b0 = blockIdx.x * 32, tid = threadIdx.x;
  for (int i = tid; i < 576; i += 256) Ws[i] = W[i];
  for (int i = tid; i < 32 * 9; i += 256) {
    const int r = i / 9, k = i % 9;
    float be = 0.f, dbe;
    if (b0 + r < nb) rbf_env_k(b_vec[b0 + r].w, rp.freq[k], rp, be, dbe);
    be_s[r][k] = be;
  }
  __syncthreads();
  for (int i = tid; i < 32 * 64; i += 256) {
    const int r = i >> 6, c = i & 63;
    if (b0 + r >= nb) continue;
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 9; k++) s = fmaf(be_s[r][k], Ws[c * 9 + k], s);
    out[(size_t)(b0 + r) * 64 + c] = s;
  }
}
void launch_bond_init(cudaStream_t st, int nb, const float4* b_vec, RadialParams rp, const float* W, float* out) {
  if (nb <= 0) return;
  k_bond_init<<<cdiv(nb, 32), 256, 0, st>>>(nb, b_vec, rp, W, out);
  B2M_CK(cudaGetLastError());
  g_launch_count++;
}

struct AngleGeom {
  float cos_raw, cc, theta, na, nb;
  float va[3], vb[3];
};
__device__ __forceinline__ AngleGeom angle_geom(const float4 a, const float4 b) {
  // compute_theta with src_bond_sign = -1 (chgnet.py:190-194; SURVEY 9): cos = (-va . vb) / (|va||vb|)
  AngleGeom g;
  g.va[0] = a.x, g.va[1] = a.y, g.va[2] = a.z;
  g.vb[0] = b.x, g.vb[1] = b.y, g.vb[2] = b.z;
  g.na = sqrtf(a.x * a.x + a.y * a.y + a.z * a.z);
  g.nb = sqrtf(b.x * b.x + b.y * b.y + b.z * b.z);
  g.cos_raw = -(a.x * b.x + a.y * b.y + a.z * b.z) / (g.na * g.nb);
  const float lo = -1.f + 1e-7f, hi = 1.f - 1e-7f;
  g.cc = fminf(fmaxf(g.cos_raw, lo), hi);
  g.theta = acosf(g.cc);
  return g;
}

// ang0[r][c] = sum_k fourier_k(theta_r) Wae[c][k]      (128 angles per block = one tile of the interleaved layout)
__global__ void __launch_bounds__(256) k_angle_init(int64_t na, const int* __restrict__ a_in,
                                                    const int* __restrict__ a_out, const float4* __restrict__ b_vec,
                                                    const float* __restrict__ fa, const float* __restrict__ Wae,
                                                    float* __restrict__ ang0, int il) {
  __shared__ float f_s[128][12];
  __shared__ float Ws[64 * 9];
  const int64_t r0 = (int64_t)blockIdx.x * 128;
  const int tid = threadIdx.x;
  for (int i = tid; i < 576; i += 256) Ws[i] = Wae[i];
  if (tid < 128) {
    const int64_t r = r0 + tid;
    if (r < na) {
      const AngleGeom g = angle_geom(b_vec[a_in[r]], b_vec[a_out[r]]);
      const float ipi = 0.318309886183790672f;
      // even columns cos(f_k theta), odd columns sin(f_k theta) (k>=1), all / pi   (SURVEY 9)
      for (int k = 0; k < 5; k++) {
        float s, c;
        sincosf(g.theta * fa[k], &s, &c);
        f_s[tid][2 * k] = c * ipi;
        if (k >= 1) f_s[tid][2 * k - 1] = s * ipi;
      }
    } else {
      for (int k = 0; k < 9; k++) f_s[tid][k] = 0.f;
    }
  }
  __syncthreads();
  for (int i = tid; i < 16 * 128; i += 256) {  // (4 columns, row): consecutive lanes = consecutive rows
    const int cq = i >> 7, r = i & 127;
    if (r0 + r >= na) continue;
    float v[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < 9; k++) {
      const float f = f_s[r][k];
#pragma unroll
      for (int j = 0; j < 4; j++) v[j] = fmaf(f, Ws[(4 * cq + j) * 9 + k], v[j]);
    }
    if (il)
      reinterpret_cast<float4*>(ang0)[(size_t)blockIdx.x * 16 * 128 + i] = make_float4(v[0], v[1], v[2], v[3]);
    else
      *reinterpret_cast<float4*>(ang0 + (size_t)(r0 + r) * 64 + 4 * cq) = make_float4(v[0], v[1], v[2], v[3]);
  }
}
void launch_angle_init(cudaStream_t st, int64_t na, const int* a_in, const int* a_out, const float4* b_vec,
                       const float* fa, const float* Wae, float* ang0, bool interleaved) {
  if (na <= 0) return;
  k_angle_init<<<cdiv(na, 128), 256, 0, st>>>(na, a_in, a_out, b_vec, fa, Wae, ang0, interleaved ? 1 : 0);
  B2M_CK(cudaGetLastError());
  g_launch_count++;
}

__global__ void k_silu(int64_t n, const float* __restrict__ pre, float* __restrict__ out) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) out[i] = silu_f(pre[i]);
}
__global__ void k_dsilu_mul(int64_t n, const float* __restrict__ pre, float* __restrict__ g) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) g[i] *= dsilu_f(pre[i]);
}
void launch_silu(cudaStream_t st, int64_t n, const float* pre, float* out) {
  if (n <= 0) return;
  k_silu<<<cdiv(n, 256), 256, 0, st>>>(n, pre, out);
  B2M_CK(cudaGetLastError());
  g_launch_count++;
}
void launch_dsilu_mul(cudaStream_t st, int64_t n, const float* pre, float* g) {
  if (n <= 0) return;
  k_dsilu_mul<<<cdiv(n, 256), 256, 0, st>>>(n, pre, g);
  B2M_CK(cudaGetLastError());
  g_launch_count++;
}
void launch_zero_rows(cudaStream_t st, float* p, int64_t nfloats) {
  if (nfloats > 0) B2M_CK(cudaMemsetAsync(p, 0, nfloats * sizeof(float), st));
}

// ============================================================================================
// atom conv: forward
// ============================================================================================
struct AtomSmemFwd {
  static constexpr int kTile = 32;  // float offset of tile (128 B for the mbarrier)
  static constexpr int kW = kTile + TM * LD;
  static constexpr int kBe = kW + 8192;
  static constexpr int kWab = kBe + TM * 12;
  static constexpr int kB2 = kWab + 576;
  static constexpr int kD = kB2 + 128;
  static constexpr int kIdx = kD + TM;
  static constexpr int kTotal = kIdx + 3 * TM;
  static constexpr size_t bytes = (size_t)kTotal * 4;
};

__global__ void __launch_bounds__(NT, 2) k_atomconv_fwd(const AtomConvArgs a) {
  extern __shared__ __align__(128) float smem[];
  uint64_t* mbar = reinterpret_cast<uint64_t*>(smem);
  float* tile = smem + AtomSmemFwd::kTile;
  float* Wsm = smem + AtomSmemFwd::kW;
  float* be_s = smem + AtomSmemFwd::kBe;
  float* wabW = smem + AtomSmemFwd::kWab;
  float* b2s = smem + AtomSmemFwd::kB2;
  float* s_d = smem + AtomSmemFwd::kD;
  int* s_src = reinterpret_cast<int*>(smem + AtomSmemFwd::kIdx);
  int* s_dst = s_src + TM;
  int* s_bond = s_dst + TM;

  const int tid = threadIdx.x;
  const int64_t e0 = (int64_t)blockIdx.x * TM;
  const int nvalid = (int)min((int64_t)TM, a.E - e0);

  if (tid < TM) {
    int src = -1, dst = -1, bond = -1;
    float d = 1.f;
    if (tid < nvalid) {
      const int64_t e = e0 + tid;
      src = a.e_src[e];
      dst = a.e_dst[e];
      bond = a.e_bond[e];
      d = a.e_vec[e].w;
    }
    s_src[tid] = src;
    s_dst[tid] = dst;
    s_bond[tid] = bond;
    s_d[tid] = d;
  }
  if (tid == 0) {
    mbar_init(mbar, 1);
    fence_barrier_init();
  }
  __syncthreads();
  // TMA row gather: A[src] (512 B per edge) straight into the tile
  if (tid == 0) mbar_expect_tx(mbar, (uint32_t)nvalid * 512u);
  if (tid < nvalid) bulk_g2s(tile + tid * LD, a.Aproj + (size_t)s_src[tid] * D2, 512u, mbar);
  stage_w(Wsm, a.W2k, 2048);
  for (int i = tid; i < 576; i += NT) wabW[i] = a.Wabw[i];
  if (tid < 128) b2s[tid] = a.b2[tid];
  {
    const int r = tid & 127, half = tid >> 7;
    const float d = s_d[r];
    const int k0 = half ? 5 : 0, k1 = half ? 9 : 5;
    for (int k = k0; k < k1; k++) {
      float be = 0.f, dbe;
      if (r < nvalid) rbf_env_k(d, a.rp.freq[k], a.rp, be, dbe);
      be_s[r * 12 + k] = be;
    }
  }
  mbar_wait(mbar, 0);
  __syncthreads();
  // pre = A[src] + C[dst] + (M.be | Q[bond]);  hid = silu(pre)
  {
    const int j = tid & 127, rh = tid >> 7;
    float Mj[9];
#pragma unroll
    for (int k = 0; k < 9; k++) Mj[k] = a.M[j * 9 + k];
    for (int i = 0; i < 64; i++) {
      const int r = rh + 2 * i;
      float v = 0.f;
      if (r < nvalid) {
        const int dst = s_dst[r], bond = s_bond[r];
        float t;
        if (a.Qproj != nullptr && bond >= 0) {
          t = a.Qproj[(size_t)bond * D2 + j];
        } else {
          t = 0.f;
#pragma unroll
          for (int k = 0; k < 9; k++) t = fmaf(be_s[r * 12 + k], Mj[k], t);
        }
        v = silu_f(tile[r * LD + j] + a.Cproj[(size_t)dst * D2 + j] + t);
      }
      tile[r * LD + j] = v;
    }
  }
  __syncthreads();
  const Map m;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; i++)
    for (int j = 0; j < 8; j++) acc[i][j] = 0.f;
  gemm64(tile, LD, m.branch * 64, Wsm + m.branch * 4096, acc, m);
#pragma unroll
  for (int i = 0; i < 8; i++)
#pragma unroll
    for (int j = 0; j < 8; j++) {
      const float u = acc[i][j] + b2s[m.branch * 64 + m.col(j)];
      acc[i][j] = m.branch == 0 ? silu_f(u) : sigm(u);
    }
  __syncthreads();
  if (m.branch == 1) {
#pragma unroll
    for (int i = 0; i < 8; i++)
#pragma unroll
      for (int j = 0; j < 8; j++) tile[m.row(i) * LD + m.col(j)] = acc[i][j];
  }
  __syncthreads();
  if (m.branch == 0) {
#pragma unroll
    for (int i = 0; i < 8; i++) {
      const int r = m.row(i);
#pragma unroll
      for (int j = 0; j < 8; j++) {
        const int c = m.col(j);
        float wab = 0.f;
#pragma unroll
        for (int k = 0; k < 9; k++) wab = fmaf(be_s[r * 12 + k], wabW[c * 9 + k], wab);
        tile[r * LD + c] = acc[i][j] * tile[r * LD + c] * wab;
      }
    }
  }
  __syncthreads();
  {
    const int c = tid & 63, part = tid >> 6;
    seg_flush(tile, LD, c, part * 32, part * 32 + 32, s_dst, a.agg, D);
  }
}

void launch_atomconv_fwd(cudaStream_t st, const AtomConvArgs& a) {
  if (a.E <= 0) return;
  static PerDeviceOnce attr;
  if (auto once_ = attr.first(); once_) {
    B2M_CK(cudaFuncSetAttribute(k_atomconv_fwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AtomSmemFwd::bytes));
  }
  k_atomconv_fwd<<<cdiv(a.E, TM), NT, AtomSmemFwd::bytes, st>>>(a);
  B2M_CK(cudaGetLastError());
  g_launch_count++;
}

// ============================================================================================
// atom conv: backward (recompute forward in-tile, then hand-derived reverse pass)
// ============================================================================================
struct AtomSmemBwd {
  static constexpr int kP = 32;
  static constexpr int kH = kP + TM * LD;
  static constexpr int kWt = kH + TM * LD;     // gwab tile [TM][LDA]
  static constexpr int kW = kWt + TM * LDA;
  static constexpr int kBe = kW + 8192;
  static constexpr int kDbe = kBe + TM * 12;
  static constexpr int kWab = kDbe + TM * 12;
  static constexpr int kM = kWab + 576;
  static constexpr int kB2 = kM + 1152;
  static constexpr int kD = kB2 + 128;
  static constexpr int kIdx = kD + TM;
  static constexpr int kTotal = kIdx + 3 * TM;
  static constexpr size_t bytes = (size_t)kTotal * 4;
};

__global__ void __launch_bounds__(NT, 1) k_atomconv_bwd(const AtomConvArgs a) {
  extern __shared__ __align__(128) float smem[];
  uint64_t* mbar = reinterpret_cast<uint64_t*>(smem);
  float* tileP = smem + AtomSmemBwd::kP;
  float* tileH = smem + AtomSmemBwd::kH;
  float* tileW = smem + AtomSmemBwd::kWt;
  float* Wsm = smem + AtomSmemBwd::kW;
  float* be_s = smem + AtomSmemBwd::kBe;
  float* dbe_s = smem + AtomSmemBwd::kDbe;
  float* wabW = smem + AtomSmemBwd::kWab;
  float* Msm = smem + AtomSmemBwd::kM;
  float* b2s = smem + AtomSmemBwd::kB2;
  float* s_d = smem + AtomSmemBwd::kD;
  int* s_src = reinterpret_cast<int*>(smem + AtomSmemBwd::kIdx);
  int* s_dst = s_src + TM;
  int* s_bond = s_dst + TM;

  const int tid = threadIdx.x;
  const int64_t e0 = (int64_t)blockIdx.x * TM;
  const int nvalid = (int)min((int64_t)TM, a.E - e0);
  const bool useQ = a.Qproj != nullptr;

  if (tid < TM) {
    int src = -1, dst = -1, bond = -1;
    float d = 1.f;
    if (tid < nvalid) {
      const int64_t e = e0 + tid;
      src = a.e_src[e];
      dst = a.e_dst[e];
      bond = a.e_bond[e];
      d = a.e_vec[e].w;
    }
    s_src[tid] = src;
    s_dst[tid] = dst;
    s_bond[tid] = bond;
    s_d[tid] = d;
  }
  if (tid == 0) {
    mbar_init(mbar, 1);
    fence_barrier_init();
  }
  __syncthreads();
  if (tid == 0) mbar_expect_tx(mbar, (uint32_t)nvalid * 512u);
  if (tid < nvalid) bulk_g2s(tileP + tid * LD, a.Aproj + (size_t)s_src[tid] * D2, 512u, mbar);
  stage_w(Wsm, a.W2k, 2048);
  for (int i = tid; i < 576; i += NT) wabW[i] = a.Wabw[i];
  for (int i = tid; i < 1152; i += NT) Msm[i] = a.M[i];
  if (tid < 128) b2s[tid] = a.b2[tid];
  {
    const int r = tid & 127, half = tid >> 7;
    const float d = s_d[r];
    const int k0 = half ? 5 : 0, k1 = half ? 9 : 5;
    for (int k = k0; k < k1; k++) {
      float be = 0.f, dbe = 0.f;
      if (r < nvalid) rbf_env_k(d, a.rp.freq[k], a.rp, be, dbe);
      be_s[r * 12 + k] = be;
      dbe_s[r * 12 + k] = dbe;
    }
  }
  mbar_wait(mbar, 0);
  __syncthreads();
  {
    const int j = tid & 127, rh = tid >> 7;
    for (int i = 0; i < 64; i++) {
      const int r = rh + 2 * i;
      float p = 0.f;
      if (r < nvalid) {
        const int dst = s_dst[r], bond = s_bond[r];
        float t;
        if (useQ && bond >= 0) {
          t = a.Qproj[(size_t)bond * D2 + j];
        } else {
          t = 0.f;
#pragma unroll
          for (int k = 0; k < 9; k++) t = fmaf(be_s[r * 12 + k], Msm[j * 9 + k], t);
        }
        p = tileP[r * LD + j] + a.Cproj[(size_t)dst * D2 + j] + t;
      }
      tileP[r * LD + j] = p;
      tileH[r * LD + j] = r < nvalid ? silu_f(p) : 0.f;
    }
  }
  __syncthreads();
  const Map m;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; i++)
    for (int j = 0; j < 8; j++) acc[i][j] = 0.f;
  gemm64(tileH, LD, m.branch * 64, Wsm + m.branch * 4096, acc, m);
#pragma unroll
  for (int i = 0; i < 8; i++)
#pragma unroll
    for (int j = 0; j < 8; j++) acc[i][j] += b2s[m.branch * 64 + m.col(j)];  // u (L) / v (G)
  __syncthreads();  // hid + W2k no longer needed
  // exchange activations between the two branches through tileH
#pragma unroll
  for (int i = 0; i < 8; i++)
#pragma unroll
    for (int j = 0; j < 8; j++) {
      const float u = acc[i][j];
      tileH[m.row(i) * LD + m.branch * 64 + m.col(j)] = m.branch == 0 ? silu_f(u) : sigm(u);
    }
  stage_w(Wsm, a.W2raw, 2048);
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const int r = m.row(i);
    const int dst = s_dst[r];
#pragma unroll
    for (int j = 0; j < 8; j++) {
      const int c = m.col(j);
      const float u = acc[i][j];
      const float po = tileH[r * LD + (1 - m.branch) * 64 + c];  // partner activation
      float g = 0.f;
      if (dst >= 0) {
        const float gm = a.gagg[(size_t)dst * D + c];
        float wab = 0.f;
#pragma unroll
        for (int k = 0; k < 9; k++) wab = fmaf(be_s[r * 12 + k], wabW[c * 9 + k], wab);
        if (m.branch == 0) {
          const float s = sigm(u);
          const float oL = u * s;
          tileW[r * LDA + c] = gm * oL * po;                 // d/d w_ab
          g = gm * po * wab * (s * (1.f + u * (1.f - s)));    // d/du
        } else {
          const float oG = sigm(u);
          g = gm * po * wab * oG * (1.f - oG);               // d/dv
        }
      } else if (m.branch == 0) {
        tileW[r * LDA + c] = 0.f;
      }
      acc[i][j] = g;
    }
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 8; i++)
#pragma unroll
    for (int j = 0; j < 8; j++) tileH[m.row(i) * LD + m.branch * 64 + m.col(j)] = acc[i][j];
  __syncthreads();
  // ghid = [gu @ W2L, gv @ W2G];  gpre = ghid * dsilu(pre)
#pragma unroll
  for (int i = 0; i < 8; i++)
    for (int j = 0; j < 8; j++) acc[i][j] = 0.f;
  gemm64(tileH, LD, m.branch * 64, Wsm + m.branch * 4096, acc, m);
#pragma unroll
  for (int i = 0; i < 8; i++)
#pragma unroll
    for (int j = 0; j < 8; j++) {
      const int idx = m.row(i) * LD + m.branch * 64 + m.col(j);
      tileP[idx] = acc[i][j] * dsilu_f(tileP[idx]);
    }
  __syncthreads();
  // ---- scatter phase ----
  {  // d E / d d_e through the radial basis (w_ab weights and, unless a bond row fed by Q, M.be)
    const int r = tid >> 1, kh = tid & 1;
    float part = 0.f;
    if (r < nvalid) {
      const int k0 = kh ? 5 : 0, k1 = kh ? 9 : 5;
      const bool viaM = !(useQ && s_bond[r] >= 0);
      for (int k = k0; k < k1; k++) {
        float s = 0.f;
        for (int c = 0; c < 64; c++) s = fmaf(tileW[r * LDA + c], wabW[c * 9 + k], s);
        if (viaM)
          for (int j = 0; j < 128; j++) s = fmaf(tileP[r * LD + j], Msm[j * 9 + k], s);
        part = fmaf(s, dbe_s[r * 12 + k], part);
      }
    }
    part += __shfl_xor_sync(0xffffffffu, part, 1);
    if (kh == 0 && r < nvalid) a.gd[e0 + r] += part;
  }
  {
    const int j = tid & 127, rh = tid >> 7;
    if (useQ && a.gQ != nullptr) {
      for (int i = 0; i < 64; i++) {
        const int r = rh + 2 * i;
        if (r < nvalid && s_bond[r] >= 0) a.gQ[(size_t)s_bond[r] * D2 + j] = tileP[r * LD + j];
      }
    }
    if (a.gA != nullptr) {
      seg_flush(tileP, LD, j, rh * 64, rh * 64 + 64, s_dst, a.gC, D2);
      for (int i = 0; i < 64; i++) {
        const int r = rh + 2 * i;
        if (r < nvalid) atomicAdd(&a.gA[(size_t)s_src[r] * D2 + j], tileP[r * LD + j]);
      }
    }
  }
}

void launch_atomconv_bwd(cudaStream_t st, const AtomConvArgs& a) {
  if (a.E <= 0) return;
  static PerDeviceOnce attr;
  if (auto once_ = attr.first(); once_) {
    B2M_CK(cudaFuncSetAttribute(k_atomconv_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AtomSmemBwd::bytes));
  }
  k_atomconv_bwd<<<cdiv(a.E, TM), NT, AtomSmemBwd::bytes, st>>>(a);
  B2M_CK(cudaGetLastError());
  g_launch_count++;
}

// ============================================================================================
// line-graph kernels: bond conv (HIDDEN) and angle update (!HIDDEN)
// ============================================================================================
struct LineSmem {
  static constexpr int kP = 32;
  static constexpr int kAng = kP + TM * LD;
  static constexpr int kW = kAng + TM * LDA;
  static constexpr int kB2 = kW + 8192;
  static constexpr int kIdx = kB2 + 128;
  static constexpr int kFwdTotal = kIdx + 3 * TM;
  static constexpr int kH = kFwdTotal;  // backward only
  static constexpr int kBwdTotal = kH + TM * LD;
  static constexpr size_t fwd_bytes = (size_t)kFwdTotal * 4;
  static constexpr size_t bwd_bytes = (size_t)kBwdTotal * 4;
};

// common prologue: indices, TMA gathers of Ha[a] rows and the tile's own angle rows, Wg staging
__device__ __forceinline__ int line_prologue(const LineArgs& a, float* smem, int64_t r0) {
  uint64_t* mbar = reinterpret_cast<uint64_t*>(smem);
  float* tileP = smem + LineSmem::kP;
  float* angT = smem + LineSmem::kAng;
  float* Wsm = smem + LineSmem::kW;
  float* b2s = smem + LineSmem::kB2;
  int* s_a = reinterpret_cast<int*>(smem + LineSmem::kIdx);
  int* s_b = s_a + TM;
  int* s_c = s_b + TM;
  const int tid = threadIdx.x;
  const int nvalid = (int)min((int64_t)TM, a.A - r0);
  if (tid < TM) {
    int ia = -1, ib = -1, ic = -1;
    if (tid < nvalid) {
      ia = a.a_in[r0 + tid];
      ib = a.a_out[r0 + tid];
      ic = a.a_ctr[r0 + tid];
    }
    s_a[tid] = ia;
    s_b[tid] = ib;
    s_c[tid] = ic;
  }
  if (tid == 0) {
    mbar_init(mbar, 1);
    fence_barrier_init();
  }
  __syncthreads();
  if (tid == 0) mbar_expect_tx(mbar, (uint32_t)nvalid * 768u);
  if (tid < nvalid) {
    bulk_g2s(tileP + tid * LD, a.Ha + (size_t)s_a[tid] * D2, 512u, mbar);
    bulk_g2s(angT + tid * LDA, a.ang + (size_t)(r0 + tid) * D, 256u, mbar);
  } else if (tid < TM) {
    for (int k = 0; k < 64; k++) angT[tid * LDA + k] = 0.f;
    for (int k = 0; k < 128; k++) tileP[tid * LD + k] = 0.f;
  }
  stage_w(Wsm, a.Wgk, 2048);
  if (tid < 128) b2s[tid] = a.b2 ? a.b2[tid] : 0.f;
  mbar_wait(mbar, 0);
  __syncthreads();
  return nvalid;
}

template <bool HIDDEN>
__global__ void __launch_bounds__(NT, 1) k_line_fwd(const LineArgs a) {
  extern __shared__ __align__(128) float smem[];
  float* tileP = smem + LineSmem::kP;
  float* angT = smem + LineSmem::kAng;
  float* Wsm = smem + LineSmem::kW;
  float* b2s = smem + LineSmem::kB2;
  int* s_a = reinterpret_cast<int*>(smem + LineSmem::kIdx);
  int* s_b = s_a + TM;
  int* s_c = s_b + TM;
  const int64_t r0 = (int64_t)blockIdx.x * TM;
  const int nvalid = line_prologue(a, smem, r0);
  (void)s_a;
  const Map m;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; i++)
    for (int j = 0; j < 8; j++) acc[i][j] = 0.f;
  gemm64(angT, LDA, 0, Wsm + m.branch * 4096, acc, m);
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const int r = m.row(i);
    const int ib = s_b[r], ic = s_c[r];
#pragma unroll
    for (int j = 0; j < 8; j++) {
      const int col = m.branch * 64 + m.col(j);
      float p = 0.f;
      if (r < nvalid) p = tileP[r * LD + col] + acc[i][j] + a.Hb[(size_t)ib * D2 + col] + a.Xc[(size_t)ic * D2 + col];
      if (HIDDEN) {
        tileP[r * LD + col] = r < nvalid ? silu_f(p) : 0.f;
      } else {
        acc[i][j] = m.branch == 0 ? silu_f(p) : sigm(p);
      }
    }
  }
  __syncthreads();
  if (HIDDEN) {
    stage_w(Wsm, a.W2k, 2048);
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 8; i++)
      for (int j = 0; j < 8; j++) acc[i][j] = 0.f;
    gemm64(tileP, LD, m.branch * 64, Wsm + m.branch * 4096, acc, m);
#pragma unroll
    for (int i = 0; i < 8; i++)
#pragma unroll
      for (int j = 0; j < 8; j++) {
        const float u = acc[i][j] + b2s[m.branch * 64 + m.col(j)];
        acc[i][j] = m.branch == 0 ? silu_f(u) : sigm(u);
      }
    __syncthreads();
  }
  if (m.branch == 1) {
#pragma unroll
    for (int i = 0; i < 8; i++)
#pragma unroll
      for (int j = 0; j < 8; j++)
        tileP[m.row(i) * LD + m.col(j)] = acc[i][j];
  }
  __syncthreads();
  if (m.branch == 0) {
#pragma unroll
    for (int i = 0; i < 8; i++) {
      const int r = m.row(i);
#pragma unroll
      for (int j = 0; j < 8; j++) {
        const int c = m.col(j);
        const float mv = acc[i][j] * tileP[r * LD + c];
        if (HIDDEN) {
          tileP[r * LD + c] = mv;
        } else if (r < nvalid) {
          a.ang_out[(size_t)(r0 + r) * D + c] = angT[r * LDA + c] + mv;
        }
      }
    }
  }
  if (HIDDEN) {
    __syncthreads();
    const int c = threadIdx.x & 63, part = threadIdx.x >> 6;
    seg_flush(tileP, LD, c, part * 32, part * 32 + 32, s_b, a.aggB, D);
  }
}

template <bool HIDDEN>
__global__ void __launch_bounds__(NT, 1) k_line_bwd(const LineArgs a) {
  extern __shared__ __align__(128) float smem[];
  float* tileP = smem + LineSmem::kP;
  float* angT = smem + LineSmem::kAng;
  float* Wsm = smem + LineSmem::kW;
  float* b2s = smem + LineSmem::kB2;
  float* tileH = smem + LineSmem::kH;
  int* s_a = reinterpret_cast<int*>(smem + LineSmem::kIdx);
  int* s_b = s_a + TM;
  int* s_c = s_b + TM;
  const int tid = threadIdx.x;
  const int64_t r0 = (int64_t)blockIdx.x * TM;
  const int nvalid = line_prologue(a, smem, r0);
  const Map m;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; i++)
    for (int j = 0; j < 8; j++) acc[i][j] = 0.f;
  gemm64(angT, LDA, 0, Wsm + m.branch * 4096, acc, m);
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const int r = m.row(i);
    const int ib = s_b[r], ic = s_c[r];
#pragma unroll
    for (int j = 0; j < 8; j++) {
      const int col = m.branch * 64 + m.col(j);
      float p = 0.f;
      if (r < nvalid) p = tileP[r * LD + col] + acc[i][j] + a.Hb[(size_t)ib * D2 + col] + a.Xc[(size_t)ic * D2 + col];
      if (HIDDEN) {
        tileP[r * LD + col] = p;
        tileH[r * LD + col] = r < nvalid ? silu_f(p) : 0.f;
      } else {
        acc[i][j] = p;
      }
    }
  }
  __syncthreads();
  if (HIDDEN) {
    stage_w(Wsm, a.W2k, 2048);
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 8; i++)
      for (int j = 0; j < 8; j++) acc[i][j] = 0.f;
    gemm64(tileH, LD, m.branch * 64, Wsm + m.branch * 4096, acc, m);
#pragma unroll
    for (int i = 0; i < 8; i++)
#pragma unroll
      for (int j = 0; j < 8; j++) acc[i][j] += b2s[m.branch * 64 + m.col(j)];
    __syncthreads();
  }
  // acc = pre-activation of the last layer of this GatedMLP (u | v).  Exchange activations.
#pragma unroll
  for (int i = 0; i < 8; i++)
#pragma unroll
    for (int j = 0; j < 8; j++) {
      const float u = acc[i][j];
      tileH[m.row(i) * LD + m.branch * 64 + m.col(j)] = m.branch == 0 ? silu_f(u) : sigm(u);
    }
  if (HIDDEN) stage_w(Wsm, a.W2raw, 2048);
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const int r = m.row(i);
    const int ib = s_b[r];
#pragma unroll
    for (int j = 0; j < 8; j++) {
      const int c = m.col(j);
      const float u = acc[i][j];
      const float po = tileH[r * LD + (1 - m.branch) * 64 + c];
      float g = 0.f;
      if (r < nvalid) {
        const float gm = HIDDEN ? a.gaggB[(size_t)ib * D + c] : a.gang[(size_t)(r0 + r) * D + c];
        if (m.branch == 0) {
          const float s = sigm(u);
          g = gm * po * (s * (1.f + u * (1.f - s)));
        } else {
          const float oG = sigm(u);
          g = gm * po * oG * (1.f - oG);
        }
      }
      acc[i][j] = g;
    }
  }
  __syncthreads();
  if (HIDDEN) {
#pragma unroll
    for (int i = 0; i < 8; i++)
#pragma unroll
      for (int j = 0; j < 8; j++) tileH[m.row(i) * LD + m.branch * 64 + m.col(j)] = acc[i][j];
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 8; i++)
      for (int j = 0; j < 8; j++) acc[i][j] = 0.f;
    gemm64(tileH, LD, m.branch * 64, Wsm + m.branch * 4096, acc, m);
#pragma unroll
    for (int i = 0; i < 8; i++)
#pragma unroll
      for (int j = 0; j < 8; j++) {
        const int idx = m.row(i) * LD + m.branch * 64 + m.col(j);
        tileP[idx] = acc[i][j] * dsilu_f(tileP[idx]);
      }
  } else {
#pragma unroll
    for (int i = 0; i < 8; i++)
#pragma unroll
      for (int j = 0; j < 8; j++) tileP[m.row(i) * LD + m.branch * 64 + m.col(j)] = acc[i][j];
  }
  __syncthreads();
  // gang += gpre @ Wg_raw   (K = 128, N = 64)
  stage_w(Wsm, a.Wgraw, 2048);
  __syncthreads();
  {
    const int rg16 = tid >> 4, cg16 = tid & 15;
    float a3[8][4];
#pragma unroll
    for (int i = 0; i < 8; i++)
      for (int j = 0; j < 4; j++) a3[i][j] = 0.f;
#pragma unroll 4
    for (int k = 0; k < 128; k++) {
      const float4 w = *reinterpret_cast<const float4*>(&Wsm[k * 64 + cg16 * 4]);
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const float av = tileP[(rg16 + 16 * i) * LD + k];
        a3[i][0] = fmaf(av, w.x, a3[i][0]);
        a3[i][1] = fmaf(av, w.y, a3[i][1]);
        a3[i][2] = fmaf(av, w.z, a3[i][2]);
        a3[i][3] = fmaf(av, w.w, a3[i][3]);
      }
    }
#pragma unroll
    for (int i = 0; i < 8; i++) {
      const int r = rg16 + 16 * i;
      if (r < nvalid) {
        float4* gp = reinterpret_cast<float4*>(&a.gang[(size_t)(r0 + r) * D + cg16 * 4]);
        float4 v = *gp;
        v.x += a3[i][0], v.y += a3[i][1], v.z += a3[i][2], v.w += a3[i][3];
        *gp = v;
      }
    }
  }
  {
    const int j = tid & 127, rh = tid >> 7;
    seg_flush(tileP, LD, j, rh * 64, rh * 64 + 64, s_b, a.gHb, D2);
    seg_flush(tileP, LD, j, rh * 64, rh * 64 + 64, s_c, a.gXc, D2);
    for (int i = 0; i < 64; i++) {
      const int r = rh + 2 * i;
      if (r < nvalid) atomicAdd(&a.gHa[(size_t)s_a[r] * D2 + j], tileP[r * LD + j]);
    }
  }
}

void launch_line_fwd(cudaStream_t st, const LineArgs& a, bool hidden) {
  if (a.A <= 0) return;
  static PerDeviceOnce attr;
  if (auto once_ = attr.first(); once_) {
    B2M_CK(cudaFuncSetAttribute(k_line_fwd<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LineSmem::fwd_bytes));
    B2M_CK(cudaFuncSetAttribute(k_line_fwd<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LineSmem::fwd_bytes));
  }
  if (hidden)
    k_line_fwd<true><<<cdiv(a.A, TM), NT, LineSmem::fwd_bytes, st>>>(a);
  else
    k_line_fwd<false><<<cdiv(a.A, TM), NT, LineSmem::fwd_bytes, st>>>(a);
  B2M_CK(cudaGetLastError());
  g_launch_count++;
}
void launch_line_bwd(cudaStream_t st, const LineArgs& a, bool hidden) {
  if (a.A <= 0) return;
  static PerDeviceOnce attr;
  if (auto once_ = attr.first(); once_) {
    B2M_CK(cudaFuncSetAttribute(k_line_bwd<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LineSmem::bwd_bytes));
    B2M_CK(cudaFuncSetAttribute(k_line_bwd<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LineSmem::bwd_bytes));
  }
  if (hidden)
    k_line_bwd<true><<<cdiv(a.A, TM), NT, LineSmem::bwd_bytes, st>>>(a);
  else
    k_line_bwd<false><<<cdiv(a.A, TM), NT, LineSmem::bwd_bytes, st>>>(a);
  B2M_CK(cudaGetLastError());
  g_launch_count++;
}

// ============================================================================================
// bond update (node-level, after the W_out GEMM):  h' = h + upd * w3b(d_b)
// ============================================================================================
// 128 bonds per block, 16-byte accesses: these are pure streaming kernels (300 MB per launch at 97 k atoms) and ran at a
// third of the HBM rate with 32 bonds per block and 4-byte accesses (profiles/r02k_kernel_shares_97k.txt)
constexpr int BNR = 128;  // bonds per block
template <int MODE>  // 0: fwd, 1: bwd (gupd, gdb), 2: h0 backward (gdb only)
__global__ void __launch_bounds__(256) k_bond_node(int nb, const float4* __restrict__ b_vec, RadialParams rp,
                                                   const float* __restrict__ W /*[64][9]*/,
                                                   const float* __restrict__ x0 /*h | gh | gh0*/,
                                                   const float* __restrict__ x1 /*upd*/, float* __restrict__ out,
                                                   float* __restrict__ gdb) {
  extern __shared__ float bn_smem[];
  float(*be_s)[12] = reinterpret_cast<float(*)[12]>(bn_smem);                 // [BNR][12]
  float(*dbe_s)[12] = reinterpret_cast<float(*)[12]>(bn_smem + BNR * 12);     // [BNR][12]
  float* Ws = bn_smem + 2 * BNR * 12;                                         // [64][9]
  float(*P)[68] = reinterpret_cast<float(*)[68]>(bn_smem + 2 * BNR * 12 + 576);  // [BNR][68]  MODE 1: gh*upd, MODE 2: gh0
  const int b0 = blockIdx.x * BNR, tid = threadIdx.x;
  for (int i = tid; i < 576; i += 256) Ws[i] = W[i];
  for (int i = tid; i < BNR * 9; i += 256) {
    const int r = i / 9, k = i % 9;
    float be = 0.f, dbe = 0.f;
    if (b0 + r < nb) rbf_env_k(b_vec[b0 + r].w, rp.freq[k], rp, be, dbe);
    be_s[r][k] = be;
    dbe_s[r][k] = dbe;
  }
  __syncthreads();
  for (int i = tid; i < BNR * 16; i += 256) {  // (row, 4 columns) per item
    const int r = i >> 4, c = (i & 15) * 4;
    float4 pv = make_float4(0.f, 0.f, 0.f, 0.f);
    if (b0 + r < nb) {
      const size_t o = (size_t)(b0 + r) * 64 + c;
      const float4 a0 = *reinterpret_cast<const float4*>(x0 + o);
      if (MODE == 2) {
        pv = a0;
      } else {
        float w[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int k = 0; k < 9; k++) {
          const float b = be_s[r][k];
#pragma unroll
          for (int j = 0; j < 4; j++) w[j] = fmaf(b, Ws[(c + j) * 9 + k], w[j]);
        }
        const float4 a1 = *reinterpret_cast<const float4*>(x1 + o);
        if (MODE == 0) {
          *reinterpret_cast<float4*>(out + o) = make_float4(a0.x + a1.x * w[0], a0.y + a1.y * w[1], a0.z + a1.z * w[2], a0.w + a1.w * w[3]);
        } else {
          *reinterpret_cast<float4*>(out + o) = make_float4(a0.x * w[0], a0.y * w[1], a0.z * w[2], a0.w * w[3]);
          pv = make_float4(a0.x * a1.x, a0.y * a1.y, a0.z * a1.z, a0.w * a1.w);
        }
      }
    }
    if (MODE != 0) *reinterpret_cast<float4*>(&P[r][c]) = pv;
  }
  if (MODE == 1 || MODE == 2) {
    __syncthreads();
    // gdb[r] += sum_k (sum_c P[r][c] W[c][k]) dbe_k : two threads per bond (k parity), partial sums combined by shuffle
    {
      const int r = tid >> 1, par = tid & 1;
      float tot = 0.f;
      for (int k = par; k < 9; k += 2) {
        float sacc = 0.f;
#pragma unroll 8
        for (int c = 0; c < 64; c++) sacc = fmaf(P[r][c], Ws[c * 9 + k], sacc);
        tot += sacc * dbe_s[r][k];
      }
      tot += __shfl_xor_sync(0xffffffffu, tot, 1);
      if (par == 0 && b0 + r < nb) gdb[b0 + r] += tot;
    }
  }
}
constexpr size_t kBondNodeSmem = (size_t)(2 * BNR * 12 + 576 + BNR * 68) * sizeof(float);
template <int MODE>
static void launch_bond_node(cudaStream_t st, int nb, const float4* b_vec, RadialParams rp, const float* W, const float* x0,
                             const float* x1, float* out, float* gdb) {
  static PerDeviceOnce attr;
  if (auto once_ = attr.first(); once_)
    B2M_CK(cudaFuncSetAttribute(k_bond_node<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBondNodeSmem));
  k_bond_node<MODE><<<cdiv(nb, BNR), 256, kBondNodeSmem, st>>>(nb, b_vec, rp, W, x0, x1, out, gdb);
  B2M_CK(cudaGetLastError());
  g_launch_count++;
}
void launch_bond_update_fwd(cudaStream_t st, int nb, const float4* b_vec, RadialParams rp3, const float* W3bw,
                            const float* h, const float* upd, float* hout) {
  if (nb <= 0) return;
  launch_bond_node<0>(st, nb, b_vec, rp3, W3bw, h, upd, hout, nullptr);
}
void launch_bond_update_bwd(cudaStream_t st, int nb, const float4* b_vec, RadialParams rp3, const float* W3bw,
                            const float* gh, const float* upd, float* gupd, float* gdb) {
  if (nb <= 0) return;
  launch_bond_node<1>(st, nb, b_vec, rp3, W3bw, gh, upd, gupd, gdb);
}
void launch_h0_bwd(cudaStream_t st, int nb, const float4* b_vec, RadialParams rp, const float* Wbe, const float* gh0,
                   float* gdb) {
  if (nb <= 0) return;
  launch_bond_node<2>(st, nb, b_vec, rp, Wbe, gh0, nullptr, nullptr, gdb);
}

// theta / Fourier backward (128 angles per block = one tile of the interleaved layout)
constexpr int ANR = 128;
__global__ void __launch_bounds__(256) k_angle_init_bwd(int64_t na, const int* __restrict__ a_in,
                                                        const int* __restrict__ a_out,
                                                        const float4* __restrict__ b_vec, const float* __restrict__ fa,
                                                        const float* __restrict__ Wae, const float* __restrict__ gang0,
                                                        float* __restrict__ gbvec, int il) {
  extern __shared__ float ab_smem[];
  float(*G)[65] = reinterpret_cast<float(*)[65]>(ab_smem);                  // [ANR][65]
  float(*gf_s)[12] = reinterpret_cast<float(*)[12]>(ab_smem + ANR * 65);    // [ANR][12]
  float* Ws = ab_smem + ANR * 65 + ANR * 12;                                // [64][9]
  const int64_t r0 = (int64_t)blockIdx.x * ANR;
  const int tid = threadIdx.x;
  for (int i = tid; i < 576; i += 256) Ws[i] = Wae[i];
  if (il) {  // tile-interleaved: float4 (c/4, row) -> consecutive lanes read consecutive rows of one column group
    const float4* g4 = reinterpret_cast<const float4*>(gang0) + (size_t)blockIdx.x * 16 * 128;
    for (int i = tid; i < 16 * ANR; i += 256) {
      const int cq = i >> 7, r = i & 127;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r0 + r < na) v = g4[i];
      G[r][4 * cq] = v.x, G[r][4 * cq + 1] = v.y, G[r][4 * cq + 2] = v.z, G[r][4 * cq + 3] = v.w;
    }
  } else {
    for (int i = tid; i < ANR * 64; i += 256) {
      const int r = i >> 6, c = i & 63;
      G[r][c] = (r0 + r < na) ? gang0[(size_t)(r0 + r) * 64 + c] : 0.f;
    }
  }
  __syncthreads();
  for (int i = tid; i < ANR * 9; i += 256) {
    const int r = i / 9, k = i % 9;
    float s = 0.f;
#pragma unroll 8
    for (int c = 0; c < 64; c++) s = fmaf(G[r][c], Ws[c * 9 + k], s);
    gf_s[r][k] = s;
  }
  __syncthreads();
  if (tid < ANR && r0 + tid < na) {
    const int64_t r = r0 + tid;
    const int ia = a_in[r], ib = a_out[r];
    const AngleGeom g = angle_geom(b_vec[ia], b_vec[ib]);
    const float ipi = 0.318309886183790672f;
    float gth = 0.f;
    for (int k = 0; k < 5; k++) {
      float s, c;
      sincosf(g.theta * fa[k], &s, &c);
      gth -= gf_s[tid][2 * k] * fa[k] * s;
      if (k >= 1) gth += gf_s[tid][2 * k - 1] * fa[k] * c;
    }
    gth *= ipi;
    const float lo = -1.f + 1e-7f, hi = 1.f - 1e-7f;
    float gcos = 0.f;
    if (g.cos_raw >= lo && g.cos_raw <= hi) gcos = -gth / sqrtf(1.f - g.cc * g.cc);
    const float inn = 1.f / (g.na * g.nb);
    const float ia2 = 1.f / (g.na * g.na), ib2 = 1.f / (g.nb * g.nb);
    for (int x = 0; x < 3; x++) {
      const float dva = -g.vb[x] * inn - g.cos_raw * g.va[x] * ia2;
      const float dvb = -g.va[x] * inn - g.cos_raw * g.vb[x] * ib2;
      atomicAdd(&gbvec[(size_t)ia * 3 + x], gcos * dva);
      atomicAdd(&gbvec[(size_t)ib * 3 + x], gcos * dvb);
    }
  }
}
constexpr size_t kAngleBwdSmem = (size_t)(ANR * 65 + ANR * 12 + 576) * sizeof(float);
void launch_angle_init_bwd(cudaStream_t st, int64_t na, const int* a_in, const int* a_out, const float4* b_vec,
                           const float* fa, const float* Wae, const float* gang0, float* gbvec, bool interleaved) {
  if (na <= 0) return;
  static PerDeviceOnce attr;
  if (auto once_ = attr.first(); once_)
    B2M_CK(cudaFuncSetAttribute(k_angle_init_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kAngleBwdSmem));
  k_angle_init_bwd<<<cdiv(na, ANR), 256, kAngleBwdSmem, st>>>(na, a_in, a_out, b_vec, fa, Wae, gang0, gbvec, interleaved ? 1 : 0);
  B2M_CK(cudaGetLastError());
  g_launch_count++;
}

// ============================================================================================
// readout
// ============================================================================================
__global__ void __launch_bounds__(256) k_rowdot(int n, const float* __restrict__ X, const float* __restrict__ w,
                                                float bias, float* __restrict__ out, double* __restrict__ sum,
                                                const int* __restrict__ type, const double* __restrict__ elem_ref,
                                                float scale) {
  // one warp per row
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  float v = 0.f;
  if (warp < n) {
    const float2 x = reinterpret_cast<const float2*>(X + (size_t)warp * 64)[lane];
    const float2 ww = reinterpret_cast<const float2*>(w)[lane];
    v = x.x * ww.x + x.y * ww.y;
  }
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __shared__ double part[8];
  double contrib = 0.0;
  if (warp < n && lane == 0) {
    v += bias;
    if (out) out[warp] = v;
    contrib = (double)scale * (double)v;
    if (elem_ref) contrib += elem_ref[type[warp]];
  }
  if (sum) {
    if (lane == 0) part[threadIdx.x >> 5] = contrib;
    __syncthreads();
    if (threadIdx.x == 0) {
      double s = 0.0;
      for (int i = 0; i < 8; i++) s += part[i];
      atomicAdd(sum, s);
    }
  }
}
void launch_rowdot(cudaStream_t st, int n, const float* X, const float* w, float bias, float* out, double* sum,
                   const int* type, const double* elem_ref, float scale) {
  if (n <= 0) return;
  k_rowdot<<<cdiv((int64_t)n * 32, 256), 256, 0, st>>>(n, X, w, bias, out, sum, type, elem_ref, scale);
  B2M_CK(cudaGetLastError());
  g_launch_count++;
}
__global__ void k_readout_seed(int n, const float* __restrict__ pre, const float* __restrict__ w, float scale,
                               float* __restrict__ g) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)n * 64) return;
  g[i] = scale * w[i & 63] * dsilu_f(pre[i]);
}
void launch_readout_seed(cudaStream_t st, int n, const float* pre, const float* w, float scale, float* g) {
  if (n <= 0) return;
  k_readout_seed<<<cdiv((int64_t)n * 64, 256), 256, 0, st>>>(n, pre, w, scale, g);
  B2M_CK(cudaGetLastError());
  g_launch_count++;
}
__global__ void k_atom_energy(int n, const float* __restrict__ e_atom, const int* __restrict__ gid,
                              const int* __restrict__ type, const double* __restrict__ elem_ref, float scale,
                              double mean_per_atom, double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  // the same terms, in the same precision, as k_rowdot's / k_tn_readout_final's contribution to the energy
  double v = (double)scale * (double)e_atom[i];
  if (elem_ref) v += elem_ref[type[i]];
  out[gid[i]] = v + mean_per_atom;
}
void launch_atom_energy(cudaStream_t st, int n_own, const float* e_atom, const int* gid, const int* type,
                        const double* elem_ref, float scale, double mean_per_atom, double* out) {
  if (n_own <= 0) return;
  k_atom_energy<<<cdiv(n_own, 256), 256, 0, st>>>(n_own, e_atom, gid, type, elem_ref, scale, mean_per_atom, out);
  B2M_CK(cudaGetLastError());
  g_launch_count++;
}

// ============================================================================================
// final geometry backward: forces and virial
// ============================================================================================
__device__ __forceinline__ void virial_reduce(const float (&v)[9], double* __restrict__ virial) {
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
__global__ void __launch_bounds__(256) k_edge_final(int64_t E, const int* __restrict__ e_src,
                                                    const int* __restrict__ e_dst, const int* __restrict__ e_bond,
                                                    const float4* __restrict__ e_vec, const int* __restrict__ gid,
                                                    const float* __restrict__ gd, const float* __restrict__ gdb,
                                                    const float* __restrict__ gbvec, float* __restrict__ forces,
                                                    double* __restrict__ virial, float* __restrict__ atom_vir) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  float vir[9];
#pragma unroll
  for (int k = 0; k < 9; k++) vir[k] = 0.f;
  int pa_dst = -1, pa_src = 0;
  if (e < E) {
    const float4 v = e_vec[e];
    float g = gd[e];
    float gx = 0.f, gy = 0.f, gz = 0.f;
    const int b = e_bond[e];
    if (b >= 0) {
      g += gdb[b];
      gx = gbvec[(size_t)b * 3], gy = gbvec[(size_t)b * 3 + 1], gz = gbvec[(size_t)b * 3 + 2];
    }
    const float s = g / v.w;
    gx += s * v.x, gy += s * v.y, gz += s * v.z;
    // vec = x_dst + off.L - x_src :  dE/dx_dst += g, dE/dx_src -= g ; F = -dE/dx   (pes.py:122-124)
    const int gdst = gid[e_dst[e]], gsrc = gid[e_src[e]];
    if constexpr (kPerAtom) pa_dst = gdst, pa_src = gsrc;
    atomicAdd(&forces[(size_t)gdst * 3], -gx);
    atomicAdd(&forces[(size_t)gdst * 3 + 1], -gy);
    atomicAdd(&forces[(size_t)gdst * 3 + 2], -gz);
    atomicAdd(&forces[(size_t)gsrc * 3], gx);
    atomicAdd(&forces[(size_t)gsrc * 3 + 1], gy);
    atomicAdd(&forces[(size_t)gsrc * 3 + 2], gz);
    // strain_bar[a][b] = sum vec[a] g[b]   (pes.py:140-145)
    vir[0] = v.x * gx, vir[1] = v.x * gy, vir[2] = v.x * gz;
    vir[3] = v.y * gx, vir[4] = v.y * gy, vir[5] = v.y * gz;
    vir[6] = v.z * gx, vir[7] = v.z * gy, vir[8] = v.z * gz;
  }
  if constexpr (kPerAtom) atom_vir_edge(atom_vir, pa_dst, pa_src, vir);
  virial_reduce(vir, virial);
}
void launch_edge_final(cudaStream_t st, int64_t E, const int* e_src, const int* e_dst, const int* e_bond,
                       const float4* e_vec, const int* gid, const float* gd, const float* gdb, const float* gbvec,
                       float* forces, double* virial, float* atom_vir) {
  if (E <= 0) return;
  if (atom_vir)
    k_edge_final<true><<<cdiv(E, 256), 256, 0, st>>>(E, e_src, e_dst, e_bond, e_vec, gid, gd, gdb, gbvec, forces,
                                                     virial, atom_vir);
  else
    k_edge_final<false><<<cdiv(E, 256), 256, 0, st>>>(E, e_src, e_dst, e_bond, e_vec, gid, gd, gdb, gbvec, forces,
                                                      virial, nullptr);
  B2M_CK(cudaGetLastError());
  g_launch_count++;
}

// kPerAtom: also W_i of both endpoints, per thread (halo bonds are few)
template <bool kPerAtom>
__global__ void __launch_bounds__(256) k_halo_bond_final(int b0, int b1, const int* __restrict__ b_src_gid,
                                                         const int* __restrict__ b_dst, const float4* __restrict__ b_vec,
                                                         const int* __restrict__ gid, const float* __restrict__ gdb,
                                                         const float* __restrict__ gbvec, float* __restrict__ forces,
                                                         double* __restrict__ virial, float* __restrict__ atom_vir) {
  const int b = b0 + blockIdx.x * blockDim.x + threadIdx.x;
  float vir[9];
#pragma unroll
  for (int k = 0; k < 9; k++) vir[k] = 0.f;
  if (b < b1) {
    const float4 v = b_vec[b];
    const float s = gdb[b] / v.w;
    const float gx = gbvec[(size_t)b * 3] + s * v.x, gy = gbvec[(size_t)b * 3 + 1] + s * v.y,
                gz = gbvec[(size_t)b * 3 + 2] + s * v.z;
    const int gdst = gid[b_dst[b]], gsrc = b_src_gid[b];
    atomicAdd(&forces[(size_t)gdst * 3], -gx);
    atomicAdd(&forces[(size_t)gdst * 3 + 1], -gy);
    atomicAdd(&forces[(size_t)gdst * 3 + 2], -gz);
    atomicAdd(&forces[(size_t)gsrc * 3], gx);
    atomicAdd(&forces[(size_t)gsrc * 3 + 1], gy);
    atomicAdd(&forces[(size_t)gsrc * 3 + 2], gz);
    vir[0] = v.x * gx, vir[1] = v.x * gy, vir[2] = v.x * gz;
    vir[3] = v.y * gx, vir[4] = v.y * gy, vir[5] = v.y * gz;
    vir[6] = v.z * gx, vir[7] = v.z * gy, vir[8] = v.z * gz;
    if constexpr (kPerAtom) {
      atom_vir_add(atom_vir, gdst, vir, 0.5f);
      atom_vir_add(atom_vir, gsrc, vir, 0.5f);
    }
  }
  virial_reduce(vir, virial);
}
void launch_halo_bond_final(cudaStream_t st, int b0, int b1, const int* b_src_gid, const int* b_dst,
                            const float4* b_vec, const int* gid, const float* gdb, const float* gbvec, float* forces,
                            double* virial, float* atom_vir) {
  if (b1 <= b0) return;
  if (atom_vir)
    k_halo_bond_final<true><<<cdiv(b1 - b0, 256), 256, 0, st>>>(b0, b1, b_src_gid, b_dst, b_vec, gid, gdb, gbvec,
                                                                forces, virial, atom_vir);
  else
    k_halo_bond_final<false><<<cdiv(b1 - b0, 256), 256, 0, st>>>(b0, b1, b_src_gid, b_dst, b_vec, gid, gdb, gbvec,
                                                                 forces, virial, nullptr);
  B2M_CK(cudaGetLastError());
  g_launch_count++;
}

// ============================================================================================
// halo pack / unpack
// ============================================================================================
__global__ void k_gather_rows(int n, int w4, const int* __restrict__ idx, const float4* __restrict__ src,
                              float4* __restrict__ dst) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)n * w4) return;
  const int r = (int)(i / w4), c = (int)(i % w4);
  dst[i] = src[(size_t)idx[r] * w4 + c];
}
__global__ void k_scatter_add_rows(int n, int w, const int* __restrict__ idx, const float* __restrict__ src,
                                   float* __restrict__ dst) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)n * w) return;
  const int r = (int)(i / w), c = (int)(i % w);
  dst[(size_t)idx[r] * w + c] += src[i];  // to-lists hold unique rows
}
void launch_gather_rows(cudaStream_t st, int n, int width, const int* idx, const float* src, float* dst) {
  if (n <= 0) return;
  const int w4 = width / 4;
  k_gather_rows<<<cdiv((int64_t)n * w4, 256), 256, 0, st>>>(n, w4, idx, reinterpret_cast<const float4*>(src),
                                                            reinterpret_cast<float4*>(dst));
  B2M_CK(cudaGetLastError());
  g_launch_count++;
}
void launch_scatter_add_rows(cudaStream_t st, int n, int width, const int* idx, const float* src, float* dst) {
  if (n <= 0) return;
  k_scatter_add_rows<<<cdiv((int64_t)n * width, 256), 256, 0, st>>>(n, width, idx, src, dst);
  B2M_CK(cudaGetLastError());
  g_launch_count++;
}

}  // namespace b2m
