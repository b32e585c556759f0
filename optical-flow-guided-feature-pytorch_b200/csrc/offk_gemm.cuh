// Gather-GEMM epilogue pieces shared by the gather-fed and the TMA-fed tcgen05 kernels.
#pragma once
#include "offk_common.cuh"

namespace offk {

// Per-row state of the epilogue (one accumulator row m).
struct EpiRow {
  int out, add;
  bool ones;
};
__device__ __forceinline__ EpiRow epi_row(const offk_gemm_t& g, int m) {
  EpiRow r;
  r.out = g.out_row[m];
  r.add = g.addend ? (g.add_row ? g.add_row[m] : r.out) : 0;
  r.ones = (m == g.a_ones_row);
  return r;
}

// Epilogue of one element D[m,n] (see offk.h for the op order).
__device__ __forceinline__ void epi_store(const offk_gemm_t& g, const EpiRow& r, int n, float v, bool atomic) {
  if (r.ones) {  // bias-gradient row of a weight-gradient GEMM
    if (g.ones_row_out) red_add_f32(g.ones_row_out + n, v);
    return;
  }
  const int oc = g.out_col[n];
  if (atomic) {
    red_add_f32(g.out + (r.out + oc), v);
    return;
  }
  if (g.bias) v += __ldg(g.bias + n);
  if (n < g.relu_pre_cols) v = fmaxf(v, 0.f);
  float gate = 1.f;
  const bool gated = g.gate && n >= g.gate_col0;
  if (gated) gate = __ldg(g.gate + (r.out + oc));
  if (gated && g.gate_first) v = gate > 0.f ? v : 0.f;
  if (g.addend) v += __ldg(g.addend + (r.add + (g.add_col ? g.add_col[n] : oc)));
  if (gated && !g.gate_first) v = gate > 0.f ? v : 0.f;
  if (g.relu_post) v = fmaxf(v, 0.f);
  g.out[r.out + oc] = v;
}

int launch_gemm_tc(const offk_gemm_t& g, cudaStream_t st, bool x3);

}  // namespace offk
