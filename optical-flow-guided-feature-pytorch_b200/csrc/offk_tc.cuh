// tcgen05 / TMEM / mbarrier / cp.async PTX wrappers and shared-memory descriptor builders shared by the two tensor-core
// GEMM kernels (gather-fed: offk_gemm_tc.cu, TMA-fed: offk_gemm_tma.cu).  sm_100a only.
#pragma once
#include "offk_gemm.cuh"

namespace offk {

constexpr int TC_BM = 128;            // UMMA M
constexpr int TC_BK = 32;             // K-block: 32 tf32 = one 128-byte swizzle row
constexpr int TC_A_BYTES = TC_BM * TC_BK * 4;  // 16 KB
constexpr int TC_MAX_STAGES = 8;

// ---------------------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "OFFK_WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra OFFK_DONE_%=;\n"
      "bra OFFK_WAIT_%=;\n"
      "OFFK_DONE_%=:\n"
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// One lane of a converged warp (elect.sync): the form the compiler recognises as "exactly one thread", so the tcgen05
// instructions under it are emitted back to back.  Under `if (lane == 0)` every tcgen05.mma was wrapped in an
// ELECT / BRA.U.ANY loop and cost ~80 clocks of issue time (profiles/timeline_*_r02q: 324 clocks per 4 MMAs), which
// bounded every main loop whose N tile is below 256.
__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "elect.sync _|p, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}
// D[tmem] (+)= A[smem desc] * B[smem desc]
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem desc]: the A operand read from tensor memory (row m of the tile = TMEM lane m, element k =
// column a_tmem + k, one 32-bit column per tf32 value: K = 8 is 8 columns -- tools/probes/tmem_a_probe.cu)
__device__ __forceinline__ void umma_tf32_ta(uint32_t tmem_d, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// all previously issued tcgen05.mma of this thread arrive on `bar` when complete
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// 32 lanes x 16 consecutive fp32 columns of this warp's TMEM quadrant
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// How many of the `room` main accumulators a 3xTF32 GEMM of `mmas` K = 8 steps per output tile uses: every partial
// accumulator costs the epilogue a full pass over tensor memory (64 B / clock: 256 clocks per 32-column chunk each,
// profiles/timeline_fp32_r02n.txt), so chains are only cut where they are long -- up to 64 MMAs per accumulator
// (K = 512).  The 490-MMA chains of motion_conv_trans_28 (K = 15680, four accumulators) meet the parity bar, so 64 does.
inline int x3_main_accumulators(int room, int mmas) {
  int want = (mmas + 63) / 64;
  if (want < 1) want = 1;
  return want < room ? want : room;
}

// The same load without the wait: the registers are undefined until tmem_ld_wait() returned (several loads may be in
// flight; one wait covers them all)
__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// registers -> 32 lanes x 16 consecutive columns of this warp's TMEM quadrant (complete after tmem_st_wait())
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Sum of `n_acc` accumulators that sit `stride` TMEM columns apart (3xTF32: the hi*hi products of K-block i go to "main"
// accumulator i % n_main, the two correction products to one more accumulator behind them).  The tensor core adds into
// its fp32 accumulator with truncation, so the error of a chain grows with its length and with the magnitude of the
// running sum: short chains for the large terms and a chain of their own for the ~2^-11 times smaller corrections keep
// the 3xTF32 result at fp32 level; the partial accumulators are added here in round-to-nearest fp32.
__device__ __forceinline__ void tmem_ld16_sum(uint32_t taddr, int n_acc, uint32_t stride, float (&v)[16]) {
  tmem_ld16(taddr, v);
  for (int a = 1; a < n_acc; ++a) {
    float t[16];
    tmem_ld16(taddr + (uint32_t)a * stride, t);
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] += t[i];
  }
}

// K-major SWIZZLE_128B shared-memory matrix descriptor (sm_100 format, cute::UMMA::SmemDescriptor):
//   [0,14) start address >> 4 | [16,30) leading byte offset >> 4 (unused for swizzled K-major: 1)
//   [32,46) stride byte offset >> 4 (1024 B between 8-row groups) | [46,48) version = 1 | [61,64) layout = 2
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// MN-major operands of kind::tf32 have exactly one legal swizzled layout: SWIZZLE_128B_BASE32B (layout type 1;
// cutlass sm100_common.inl: "for mn-major tf32 operands, SW128_32B is the only available smem layout").
// The tile is a grid of 512-byte atoms: 32 consecutive m|n (one 128-byte row) times 4 consecutive k, with the
// 32-byte units of a row XOR-ed by the row index (byte-address bits [5,7) ^= bits [7,9), cute Swizzle<2,5,2>).
// LBO = byte stride between atoms along m|n, SBO = byte stride between 4-k groups
// (cute::UMMA::make_umma_desc<Major::MN>: leading_byte_offset = MN-atom stride, stride_byte_offset = k-group stride).
__device__ __forceinline__ uint64_t make_smem_desc_mn(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)1 << 61;
  return d;
}
// Instruction descriptor (cute::UMMA::InstrDescriptor): D=f32 [4,6)=1, A=tf32 [7,10)=2, B=tf32 [10,13)=2,
// A / B major at bits 15 / 16 (0 = K-major, 1 = MN-major), N>>3 at [17,23), M>>4 at [24,29).
__device__ __forceinline__ uint32_t make_idesc_tf32(int n, bool a_mn, bool b_mn) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
         ((uint32_t)(n >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
}
// byte offset of (16-byte chunk `c` of 4 consecutive m|n, column k) inside an MN-major SWIZZLE_128B_BASE32B tile whose
// 512-byte atoms are ordered [4-k group][atom along m|n]; atoms_mn = number of 32-wide atoms along m|n.
__device__ __forceinline__ uint32_t swz_mn(int c, int k, int atoms_mn) {
  const int kl = k & 3, cc = c & 7;
  return (uint32_t)((((k >> 2) * atoms_mn + (c >> 3)) << 9) + (kl << 7) + (((((cc >> 1) ^ kl) << 1) | (cc & 1)) << 4));
}
// byte offset of (row r, 16-byte chunk c) inside a K-major SWIZZLE_128B tile (8-row atoms of 1024 B)
__device__ __forceinline__ uint32_t swz(int r, int c) {
  return (uint32_t)((r >> 3) * 1024 + (r & 7) * 128 + ((c ^ (r & 7)) << 4));
}
__device__ __forceinline__ void sts128(uint32_t addr, float a, float b, float c, float d) {
  asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ float lds32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts32(uint32_t addr, float a) {
  asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(a) : "memory");
}

// 16-byte asynchronous global->shared copy; src_bytes = 0 zero-fills the destination (padding / out-of-box taps)
__device__ __forceinline__ void cp_async16_ca(uint32_t dst, const float* src, uint32_t src_bytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async16_cg(uint32_t dst, const float* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
// this thread's arrival on `bar` fires once all its prior cp.async have landed (counts as one expected arrival)
__device__ __forceinline__ void cp_async_mbar_arrive_noinc(uint32_t bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}


__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ---------------------------------------------------------------------------- 3xTF32 (OFFK_PREC_TF32X3)
// tcgen05.mma kind::tf32 reads the top 19 bits of each fp32 operand word (sign, 8 exponent, 10 mantissa bits: the low
// 13 mantissa bits are ignored).  The error-compensated mode therefore keeps the operand tile as it landed ("hi": the
// tensor core truncates it by itself) and adds a second tile "lo" = tf32(x - trunc(x)) -- the part the truncation
// dropped, rounded to nearest so that its own 11 significant bits are unbiased -- and issues
//   D += A_lo * B_hi + A_hi * B_lo + A_hi * B_hi
// into the same fp32 TMEM accumulator: per-product relative error ~2^-21 instead of tf32's 2^-10 (fp32: 2^-24).
__device__ __forceinline__ float tf32_lo(float x) {
  const float hi = __uint_as_float(__float_as_uint(x) & 0xFFFFE000u);
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x - hi));
  return __uint_as_float(r);
}
// lo tile of 4 consecutive operand words: read the hi tile at `addr`, write the residual `lo_off` bytes further
__device__ __forceinline__ void split_chunk(uint32_t addr, uint32_t lo_off) {
  const float4 v = lds128(addr);
  asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(addr + lo_off), "f"(tf32_lo(v.x)), "f"(tf32_lo(v.y)),
               "f"(tf32_lo(v.z)), "f"(tf32_lo(v.w))
               : "memory");
}

__device__ __forceinline__ float4 ldg128(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float4 f4zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ float4 f4relu(float4 v) {
  return make_float4(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f), fmaxf(v.z, 0.f), fmaxf(v.w, 0.f));
}


// ---------------------------------------------------------------------------- epilogue
// Row-contiguous outputs (offk.h: out_vec = 2; weight gradients dW[n][m]): the 256 epilogue threads transpose 32-column
// chunks of the accumulator through shared memory ([column][row], pitch 132 floats, two buffers at `stg0`: 33792 bytes) so
// that one lane holds 4 consecutive rows of one column and adds them with ONE red.global.add.v4 -- scalar reds cost
// ~1.3 clocks per element and SM (a 128 x 160 tile: 14-17 thousand clocks, profiles/timeline_fp32_r02z.txt), more than
// the main loop of most weight-gradient tiles.  quad = TMEM lane quadrant of the warp, half = which 16 columns of a chunk
// it drains, ew = 0..7 (columns ew, ew + 8, ... of the chunk are added by this warp); barrier 1 is shared by the 256.
constexpr int EPI_T_PITCH = TC_BM + 4;
__device__ __forceinline__ void epi_rows_contiguous(const offk_gemm_t& g, uint32_t stg0, uint32_t tmem_d, int n_acc,
                                                    uint32_t acc_stride, int bn, int m0, int n0, int quad, int half, int ew,
                                                    int lane, bool atomic) {
  const int trow = quad * 32 + lane;
  const int nchunks = (bn + 31) >> 5;
  const int m = m0 + 4 * lane;                                   // first of the 4 rows this lane stores
  const bool all4 = m + 3 < g.M && !(g.a_ones_row >= m && g.a_ones_row < m + 4);
  const int orow = m < g.M ? __ldg(g.out_row + m) : 0;
  for (int c = 0; c < nchunks; ++c) {
    const uint32_t stg = stg0 + (uint32_t)(c & 1) * (32 * EPI_T_PITCH * 4);
    if (c * 32 + half * 16 < bn) {
      float v[16];
      tmem_ld16_sum(tmem_d + ((uint32_t)(quad * 32) << 16) + (uint32_t)(c * 32 + half * 16), n_acc, acc_stride, v);
#pragma unroll
      for (int j = 0; j < 16; ++j) sts32(stg + (uint32_t)((half * 16 + j) * EPI_T_PITCH + trow) * 4, v[j]);
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      const int col = ew + 8 * jj, n = n0 + c * 32 + col;
      if (n >= g.N || c * 32 + col >= bn || m >= g.M) continue;
      const float4 v = lds128(stg + (uint32_t)(col * EPI_T_PITCH + 4 * lane) * 4);
      const int oc = __ldg(g.out_col + n);
      if (all4) {
        float* o = g.out + (orow + oc);
        if (atomic) asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(o), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
        else *reinterpret_cast<float4*>(o) = v;
      } else {                                                   // the tile's last rows: bias-gradient row, end of M
        const float e[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int mm = m + k;
          if (mm >= g.M) continue;
          if (mm == g.a_ones_row) {
            if (g.ones_row_out) red_add_f32(g.ones_row_out + n, e[k]);
          } else if (atomic) {
            red_add_f32(g.out + (__ldg(g.out_row + mm) + oc), e[k]);
          } else {
            g.out[__ldg(g.out_row + mm) + oc] = e[k];
          }
        }
      }
    }
  }
}

// The epilogue of offk.h on 4 consecutive columns n..n+3 of one accumulator row (out_vec = 1): the float4 form of
// epi_store's op chain.  The caller fetches the operands -- bias4, gate values t and add4 are 0, 1 and 0 where absent --
// and gated = the gate applies to these columns.
__device__ __forceinline__ float4 epi_act4(const offk_gemm_t& g, float4 v, int n, const float4& bias4, const float4& t,
                                           const float4& add4, bool gated) {
  v.x += bias4.x; v.y += bias4.y; v.z += bias4.z; v.w += bias4.w;
  if (n < g.relu_pre_cols) v = f4relu(v);               // relu_pre_cols is a multiple of 4 on this path
  if (gated && g.gate_first) {
    v.x = t.x > 0.f ? v.x : 0.f; v.y = t.y > 0.f ? v.y : 0.f; v.z = t.z > 0.f ? v.z : 0.f; v.w = t.w > 0.f ? v.w : 0.f;
  }
  v.x += add4.x; v.y += add4.y; v.z += add4.z; v.w += add4.w;
  if (gated && !g.gate_first) {
    v.x = t.x > 0.f ? v.x : 0.f; v.y = t.y > 0.f ? v.y : 0.f; v.z = t.z > 0.f ? v.z : 0.f; v.w = t.w > 0.f ? v.w : 0.f;
  }
  if (g.relu_post) v = f4relu(v);
  return v;
}


}  // namespace offk
