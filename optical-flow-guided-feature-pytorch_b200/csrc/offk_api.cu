// extern "C" surface of liboffk.so that is not tied to one kernel family.
#include "offk_gemm.cuh"

namespace offk {
thread_local char g_err[512] = "";

int sm_count() {
  static int cached = 0;
  if (!cached) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&cached, cudaDevAttrMultiProcessorCount, dev);
  }
  return cached;
}
}  // namespace offk

using namespace offk;

extern "C" int offk_version(void) { return OFFK_VERSION; }
extern "C" const char* offk_last_error_string(void) { return g_err; }

extern "C" int offk_device_info(int* sm_count_out, int* cc_major, int* cc_minor, long long* l2_bytes) {
  int dev = 0;
  if (int e = cuda_check(cudaGetDevice(&dev), "cudaGetDevice")) return e;
  cudaDeviceProp prop;
  if (int e = cuda_check(cudaGetDeviceProperties(&prop, dev), "cudaGetDeviceProperties")) return e;
  if (sm_count_out) *sm_count_out = prop.multiProcessorCount;
  if (cc_major) *cc_major = prop.major;
  if (cc_minor) *cc_minor = prop.minor;
  if (l2_bytes) *l2_bytes = (long long)prop.l2CacheSize;
  return 0;
}

extern "C" int offk_drop_keep_host(uint64_t seed, uint64_t idx, float drop_p) {
  return drop_keep(seed, idx, drop_threshold16(drop_p)) ? 1 : 0;
}

extern "C" int offk_gather_gemm(const offk_gemm_t* g, int precision, void* stream) {
  OFFK_REQUIRE(g != nullptr, "gather_gemm: null descriptor");
  OFFK_REQUIRE(g->M > 0 && g->N > 0 && g->K > 0, "gather_gemm: empty problem M=%d N=%d K=%d", g->M, g->N, g->K);
  OFFK_REQUIRE(g->a_src && g->a_row && g->a_col && g->b_src && g->b_row && g->b_col, "gather_gemm: operand tables");
  OFFK_REQUIRE(g->out && g->out_row && g->out_col, "gather_gemm: output tables");
  OFFK_REQUIRE(g->a_ones_row < 0 || g->a_ones_row < g->M, "gather_gemm: a_ones_row out of range");
  OFFK_REQUIRE(g->a_mode >= OFFK_LOAD_VEC_K && g->a_mode <= OFFK_LOAD_VEC_ROW && g->b_mode >= OFFK_LOAD_VEC_K &&
               g->b_mode <= OFFK_LOAD_VEC_ROW, "gather_gemm: bad load mode");
  OFFK_REQUIRE((reinterpret_cast<uintptr_t>(g->a_src) & 15u) == 0, "gather_gemm: a_src alignment");
  OFFK_REQUIRE((reinterpret_cast<uintptr_t>(g->b_src) & 15u) == 0, "gather_gemm: b_src alignment");
  if (g->a_mode == OFFK_LOAD_VEC_K || g->b_mode == OFFK_LOAD_VEC_K) OFFK_REQUIRE((g->K & 3) == 0, "gather_gemm: VEC_K needs K %% 4 == 0");
  if (g->out_vec == 1) OFFK_REQUIRE((g->N & 3) == 0 && (reinterpret_cast<uintptr_t>(g->out) & 15u) == 0, "gather_gemm: out_vec alignment");
  if (g->out_vec == 2)
    OFFK_REQUIRE((reinterpret_cast<uintptr_t>(g->out) & 15u) == 0 && !g->bias && !g->gate && !g->addend && !g->relu_pre_cols && !g->relu_post,
                 "gather_gemm: out_vec = 2 needs a 16-byte aligned `out` and a plain epilogue");
  if (precision == OFFK_PREC_TF32) return launch_gemm_tc(*g, as_stream(stream), false);
  if (precision == OFFK_PREC_TF32X3) return launch_gemm_tc(*g, as_stream(stream), true);
  return fail(OFFK_E_BADARG, "gather_gemm: unknown precision %d", precision);
}
