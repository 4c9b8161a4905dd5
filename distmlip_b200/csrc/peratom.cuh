// Per-atom virial accumulation, shared by the per-atom instances of the edge-final kernels (kernels.cu, kernels_tn.cu).
//   W_i[a][b] = 1/2 sum_{e : src(e)=i or dst(e)=i} vec_e[a] g_e[b]      (g_e = dE/dvec_e; not symmetrised)
// Rows are [N][kAtomVirW] f32, the 9 entries row-major followed by 3 zeros of padding (48 B): one row takes three
// red.global.add.v4.f32.
#pragma once
#include "tc_common.cuh"

namespace b2m {

__device__ __forceinline__ void atom_vir_add(float* __restrict__ W, int gid, const float (&v)[9], float s) {
  float* p = W + (size_t)gid * kAtomVirW;
  red_add_v4(p, s * v[0], s * v[1], s * v[2], s * v[3]);
  red_add_v4(p + 4, s * v[4], s * v[5], s * v[6], s * v[7]);
  red_add_v4(p + 8, s * v[8], 0.f, 0.f, 0.f);
}

// Edges are CSR by owned destination, so a warp's lanes mostly share gdst: the destination halves are summed over each
// run of equal gdst inside the warp (segmented suffix scan, the run's first lane ends with the run's sum) and issued once
// per run; the source halves stay per edge.  gdst < 0 marks a lane without an edge (v must be zero there).  All 32 lanes
// of the warp must call it.
__device__ __forceinline__ void atom_vir_edge(float* __restrict__ W, int gdst, int gsrc, const float (&v)[9]) {
  const int lane = threadIdx.x & 31;
  const int prev = __shfl_up_sync(0xffffffffu, gdst, 1);
  const unsigned heads = __ballot_sync(0xffffffffu, lane == 0 || prev != gdst);
  const unsigned later = heads & ~((2u << lane) - 1u);  // run heads above this lane (lane 31: none)
  const int end = later ? __ffs(later) - 2 : 31;        // last lane of this lane's run
  float r[9];
#pragma unroll
  for (int k = 0; k < 9; k++) r[k] = v[k];
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
#pragma unroll
    for (int k = 0; k < 9; k++) {
      const float x = __shfl_down_sync(0xffffffffu, r[k], o);
      if (lane + o <= end) r[k] += x;
    }
  }
  if (gdst < 0) return;
  if ((heads >> lane) & 1u) atom_vir_add(W, gdst, r, 0.5f);
  atom_vir_add(W, gsrc, v, 0.5f);
}

}  // namespace b2m
