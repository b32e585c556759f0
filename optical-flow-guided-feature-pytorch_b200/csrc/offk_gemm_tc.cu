// tcgen05 gather-GEMM (OFFK_PREC_TF32 / OFFK_PREC_TF32X3) for sm_100a: the operands that no TMA tensor map describes
// (offk.h lists what the engine launches it for).
//
//   D[128 x BN] (fp32, TMEM) += A[128 x 32] (tf32, smem) * B[BN x 32]^T (tf32, smem)   per K-block
//
// Warp roles (288 threads):
//   warps 0-7  producers: gather A and B through the index tables with 16-byte cp.async straight into
//              shared memory, never through registers.  OFFK_LOAD_VEC_K (source contiguous along k) fills
//              the canonical K-major SWIZZLE_128B tile; OFFK_LOAD_VEC_ROW (source contiguous along m / n)
//              fills the canonical MN-major SWIZZLE_128B tile and the instruction descriptor marks that
//              operand MN-major, so no transpose is ever executed.  Producers then fence to the async
//              proxy and arrive on the stage's "full" mbarrier.  After the main loop the same
//              warps run the epilogue: tcgen05.ld the accumulator rows out of TMEM, apply
//              bias / ReLU / gate / residual, store coalesced along pixels (or atomically for
//              split-K and weight gradients).
//   warp 8     allocates TMEM; one elected lane waits on "full", issues 4 x tcgen05.mma
//              (kind::tf32, M=128, N=BN, K=8) per stage and tcgen05.commit's to the stage's "empty"
//              mbarrier (and to "accum_full" after the last K-block).
// One output tile per CTA; two CTAs co-reside per SM (<=110 KB smem, <=256 TMEM columns each) so one
// CTA's epilogue overlaps the other's main loop.
#include "offk_tc.cuh"

namespace offk {

constexpr int TC_PRODUCERS = 256;     // producer / epilogue threads (8 warps)
constexpr int TC_THREADS = TC_PRODUCERS + 32;

// ---------------------------------------------------------------------------- producers
struct TcShared {
  uint64_t full[TC_MAX_STAGES];
  uint64_t empty[TC_MAX_STAGES];
  uint64_t accum_full;
  uint32_t tmem_base;
};

// ---- table contract of the tensor-core path (the host pads, the kernel never bounds-checks an index):
//   a_row : ceil(M/128)*128 entries, a_col : ceil(K/32)*32 + 64 entries; padding entries have y = -16384, so the
//           box test (always on: a_h >= 1, 32767 = "no box") rejects them and the element is 0;
//   b_row : ceil(N/256)*256 entries, b_col : ceil(K/32)*32 + 64 entries; padding entries are 0 (they read real,
//           finite data that only ever meets a zero of A or lands in an accumulator column that is never stored).
__device__ __forceinline__ bool box_ok(const offk_gemm_t& g, uint32_t ryx, uint32_t cyx) {
  // packed (x << 16 | y) int16 pairs; per-half add without carry between halves
  const int y = (int)(short)(ryx & 0xFFFFu) + (int)(short)(cyx & 0xFFFFu);
  const int x = ((int)ryx >> 16) + ((int)cyx >> 16);
  return (unsigned)y < (unsigned)g.a_h && (unsigned)x < (unsigned)g.a_w;
}
struct Idx2 {           // offk_idx_t viewed as two 32-bit words
  int off;
  uint32_t yx;
};
__device__ __forceinline__ Idx2 ld_idx(const offk_idx_t* p) {
  const uint2 v = __ldg(reinterpret_cast<const uint2*>(p));
  return Idx2{(int)v.x, v.y};
}

// ============================ A operand (validity box, ones row)
// VEC_K  : thread = (row (tid>>3)+32i, chunk tid&7), i < 4.   cp.async, zero-fill for invalid.   K-major tile.
// VEC_ROW: thread = (row-quad tid&31, column (tid>>5)+8i), i < 4.   cp.async, zero-fill.          MN-major tile.
template <int MODE>
struct LoaderA {
  static_assert(MODE == OFFK_LOAD_VEC_K || MODE == OFFK_LOAD_VEC_ROW, "gather-GEMM operands are 16-byte vector loads");
  Idx2 r[4];
  uint32_t dst[4];
  uint32_t ones;       // VEC_K: bit i; VEC_ROW: bit 0
  Idx2 c_cur[4], c_nxt[4];
  __device__ __forceinline__ void init(const offk_gemm_t& g, int m0, int tid) {
    const int warp = tid >> 5, lane = tid & 31;
    ones = 0;
    if (MODE == OFFK_LOAD_VEC_K) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int tr = (tid >> 3) + 32 * i;
        r[i] = ld_idx(g.a_row + m0 + tr);
        dst[i] = swz(tr, tid & 7);
        ones |= (m0 + tr == g.a_ones_row ? 1u : 0u) << i;
      }
    } else {
      r[0] = ld_idx(g.a_row + m0 + 4 * lane);
#pragma unroll
      for (int i = 0; i < 4; ++i) dst[i] = swz_mn(lane, warp + 8 * i, TC_BM / 32);
      ones = (m0 + 4 * lane == g.a_ones_row) ? 1u : 0u;
    }
  }
  __device__ __forceinline__ void fetch_cols(const offk_gemm_t& g, int k0, int tid, Idx2 (&c)[4]) const {
    if (MODE == OFFK_LOAD_VEC_K) {
      c[0] = ld_idx(g.a_col + k0 + 4 * (tid & 7));
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) c[i] = ld_idx(g.a_col + k0 + (tid >> 5) + 8 * i);
    }
  }
  // 3xTF32: residuals of the chunks THIS thread copied (they have landed: cp.async.wait_group)
  __device__ __forceinline__ void split_async(uint32_t tile, uint32_t lo_off) const {
#pragma unroll
    for (int i = 0; i < 4; ++i) split_chunk(tile + dst[i], lo_off);
  }
  // straight to shared memory.  Returns true when st.shared was used (ones row).
  __device__ __forceinline__ bool issue_async(const offk_gemm_t& g, const Idx2 (&c)[4], uint32_t tile) const {
    bool stored = false;
    if (MODE == OFFK_LOAD_VEC_K) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const uint32_t d = tile + dst[i];
        if ((ones >> i) & 1u) {
          const float one = (short)(c[0].yx & 0xFFFFu) > -8192 ? 1.f : 0.f;
          sts128(d, one, one, one, one);
          stored = true;
        } else {
          const bool ok = box_ok(g, r[i].yx, c[0].yx);
          cp_async16_ca(d, ok ? g.a_src + (r[i].off + c[0].off) : g.a_src, ok ? 16u : 0u);
        }
      }
    } else {   // VEC_ROW: 4 consecutive rows of column k = (tid>>5)+8i
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const uint32_t d = tile + dst[i];
        if (ones) {   // the all-ones row heads its own row-quad: (1,0,0,0) for real columns
          sts128(d, (short)(c[i].yx & 0xFFFFu) > -8192 ? 1.f : 0.f, 0.f, 0.f, 0.f);
          stored = true;
        } else {
          const bool ok = box_ok(g, r[0].yx, c[i].yx);
          cp_async16_cg(d, ok ? g.a_src + (r[0].off + c[i].off) : g.a_src, ok ? 16u : 0u);
        }
      }
    }
    return stored;
  }
  static constexpr bool kMN = (MODE == OFFK_LOAD_VEC_ROW);
  __device__ __forceinline__ void prologue(const offk_gemm_t& g, int k_first, int tid) { fetch_cols(g, k_first, tid, c_cur); }
  __device__ __forceinline__ void pre_wait(const offk_gemm_t& g, int k0, int tid) { fetch_cols(g, k0 + TC_BK, tid, c_nxt); }
  __device__ __forceinline__ bool post_wait(const offk_gemm_t& g, uint32_t tile) {
    const bool stored = issue_async(g, c_cur, tile);
#pragma unroll
    for (int q = 0; q < 4; ++q) c_cur[q] = c_nxt[q];
    return stored;
  }
};

// ============================ B operand (plain gather, up to 256 rows)
template <int MODE>
struct LoaderB {
  static_assert(MODE == OFFK_LOAD_VEC_K || MODE == OFFK_LOAD_VEC_ROW, "gather-GEMM operands are 16-byte vector loads");
  int r[8];            // VEC_K: rows (tid>>3)+32i, i<8;  VEC_ROW: row-quads of pass 0 / pass 1 in r[0], r[1]
  uint32_t dst[8];
  int c_cur[4], c_nxt[4];
  int bn;
  __device__ __forceinline__ void init(const offk_gemm_t& g, int n0, int bn_, int tid) {
    bn = bn_;
    const int warp = tid >> 5, lane = tid & 31;
    if (MODE == OFFK_LOAD_VEC_K) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int tr = (tid >> 3) + 32 * i;
        r[i] = __ldg(g.b_row + n0 + (tr < bn ? tr : 0));
        dst[i] = swz(tr, tid & 7);
      }
    } else {
      // MN-major tile: thread = (row-quad lane of pass p, column warp+8i); atoms ordered [k-group][n-atom]
      const int atoms = (bn + 31) >> 5;
#pragma unroll
      for (int p = 0; p < 2; ++p) {
        const int tr = 128 * p + 4 * lane;
        r[p] = __ldg(g.b_row + n0 + (tr < bn ? tr : 0));
        dst[p] = swz_mn(32 * p + lane, warp, atoms);     // + i * atoms * 1024 for column warp + 8i
      }
      dst[2] = (uint32_t)atoms << 10;
    }
  }
  __device__ __forceinline__ void fetch_cols(const offk_gemm_t& g, int k0, int tid, int (&c)[4]) const {
    if (MODE == OFFK_LOAD_VEC_K) {
      c[0] = __ldg(g.b_col + k0 + 4 * (tid & 7));
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) c[i] = __ldg(g.b_col + k0 + (tid >> 5) + 8 * i);
    }
  }
  // 3xTF32: residuals of the chunks THIS thread copied (same predicates as post_wait)
  __device__ __forceinline__ void split_async(uint32_t tile, int tid, uint32_t lo_off) const {
    if (MODE == OFFK_LOAD_VEC_K) {
      const int nrow = (bn + 31) >> 5;
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if (i < nrow && (tid >> 3) + 32 * i < bn) split_chunk(tile + dst[i], lo_off);
    } else {
#pragma unroll
      for (int p = 0; p < 2; ++p)
        if (128 * p + 4 * (tid & 31) < bn) {
#pragma unroll
          for (int i = 0; i < 4; ++i) split_chunk(tile + dst[p] + i * dst[2], lo_off);
        }
    }
  }
  static constexpr bool kMN = (MODE == OFFK_LOAD_VEC_ROW);
  __device__ __forceinline__ void prologue(const offk_gemm_t& g, int k_first, int tid) { fetch_cols(g, k_first, tid, c_cur); }
  __device__ __forceinline__ void pre_wait(const offk_gemm_t& g, int k0, int tid) { fetch_cols(g, k0 + TC_BK, tid, c_nxt); }
  __device__ __forceinline__ void post_wait(const offk_gemm_t& g, uint32_t tile, int tid) {
    if (MODE == OFFK_LOAD_VEC_K) {
      const int nrow = (bn + 31) >> 5;          // 32 rows per i
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if (i < nrow && (tid >> 3) + 32 * i < bn) cp_async16_cg(tile + dst[i], g.b_src + (r[i] + c_cur[0]), 16u);
    } else {
#pragma unroll
      for (int p = 0; p < 2; ++p)
        if (128 * p + 4 * (tid & 31) < bn) {
#pragma unroll
          for (int i = 0; i < 4; ++i) cp_async16_cg(tile + dst[p] + i * dst[2], g.b_src + (r[p] + c_cur[i]), 16u);
        }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) c_cur[q] = c_nxt[q];
  }
};

// ---------------------------------------------------------------------------- kernel
// X3 = OFFK_PREC_TF32X3: every stage holds [A | B | A_lo | B_lo].  Each producer thread turns the chunks it copied itself
// into their tf32 residuals (offk_tc.cuh) once its cp.async groups have landed -- `la` K-blocks behind the issue front --
// and only then arrives on "full"; the MMA thread issues three MMAs per K = 8 step.
template <int A_MODE, int B_MODE, bool X3>
__global__ void __launch_bounds__(TC_THREADS, 2)
gather_gemm_tc_kernel(const offk_gemm_t g, int bn, int stages, int kb_per_split, int tmem_cols, int la, int n_main) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // carve: [stages x (A 16 KB | B bn*128)] then the barrier block
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t b_bytes = ((uint32_t)(bn + 31) >> 5) << 12;      // whole 32-row groups (MN-major atoms are 32 wide)
  const uint32_t hi_bytes = TC_A_BYTES + b_bytes;
  const uint32_t stage_bytes = X3 ? 2u * hi_bytes : hi_bytes;
  TcShared* sh = reinterpret_cast<TcShared*>(smem_raw + (smem_base - smem_u32(smem_raw)) + stages * stage_bytes);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int m0 = blockIdx.x * TC_BM, n0 = blockIdx.y * bn;
  const int num_kb_total = (g.K + TC_BK - 1) / TC_BK;
  const int kb_begin = blockIdx.z * kb_per_split;
  const int kb_end = min(num_kb_total, kb_begin + kb_per_split);
  const int nkb = kb_end - kb_begin;

  if (tid == 0) {
    for (int s = 0; s < stages; ++s) {
      mbar_init(smem_u32(&sh->full[s]), TC_PRODUCERS);
      mbar_init(smem_u32(&sh->empty[s]), 1);
    }
    mbar_init(smem_u32(&sh->accum_full), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 8) tmem_alloc(smem_u32(&sh->tmem_base), (uint32_t)tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_d = sh->tmem_base;
  // programmatic dependent launch (see offk_gemm_tma.cu): the prologue above may overlap the previous kernel's tail
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  if (warp < 8) {
    // ================= producers =================
    // both operands go global->smem with cp.async (up to `stages` K-blocks in flight, no registers); the column table
    // entries of the NEXT K-block are loaded before the empty-wait of this one.
    LoaderA<A_MODE> pa;
    LoaderB<B_MODE> pb;
    pa.init(g, m0, tid);
    pb.init(g, n0, bn, tid);
    if (nkb > 0) {
      pa.prologue(g, kb_begin * TC_BK, tid);
      pb.prologue(g, kb_begin * TC_BK, tid);
    }
    int s = 0;
    uint32_t parity = 1;                                       // empty-barrier parity of the current round
    if (X3) {
      // issue front at K-block `it`, residual + hand-over `la` K-blocks behind it (la < stages, so the empty-wait of
      // iteration `it` only ever needs hand-overs of earlier iterations)
      int s2 = 0;
      for (int it = 0; it < nkb + la; ++it) {
        if (it < nkb) {
          const int k0 = (kb_begin + it) * TC_BK;
          const uint32_t a_base = smem_base + s * stage_bytes;
          pa.pre_wait(g, k0, tid);
          pb.pre_wait(g, k0, tid);
          mbar_wait(smem_u32(&sh->empty[s]), parity);
          pa.post_wait(g, a_base);
          pb.post_wait(g, a_base + TC_A_BYTES, tid);
          if (++s == stages) { s = 0; parity ^= 1u; }
        }
        cp_async_commit();                                     // one group per iteration (empty past the last K-block)
        if (it >= la) {
          if (la == 1) cp_async_wait_group<1>(); else if (la == 2) cp_async_wait_group<2>(); else cp_async_wait_group<3>();
          const uint32_t a_base = smem_base + s2 * stage_bytes;
          pa.split_async(a_base, hi_bytes);
          pb.split_async(a_base + TC_A_BYTES, tid, hi_bytes);
          fence_proxy_async_smem();                            // generic-proxy st.shared -> visible to the tensor core
          mbar_arrive(smem_u32(&sh->full[s2]));
          if (++s2 == stages) s2 = 0;
        }
      }
    } else
    for (int i = 0; i < nkb; ++i) {
      const int k0 = (kb_begin + i) * TC_BK;
      const uint32_t a_base = smem_base + s * stage_bytes;
      const uint32_t b_base = a_base + TC_A_BYTES;
      pa.pre_wait(g, k0, tid);
      pb.pre_wait(g, k0, tid);
      mbar_wait(smem_u32(&sh->empty[s]), parity);              // slot free (first round passes at once)
      const bool stored = pa.post_wait(g, a_base);
      pb.post_wait(g, b_base, tid);
      if (stored) fence_proxy_async_smem();   // ones row: generic-proxy st.shared -> visible to the tensor core (async proxy)
      cp_async_mbar_arrive_noinc(smem_u32(&sh->full[s]));
      if (++s == stages) { s = 0; parity ^= 1u; }
    }
  } else {
    {
      // ================= MMA issuer (converged warp; one elected lane issues: elect_one_sync in offk_tc.cuh) =================
      constexpr bool A_MN = LoaderA<A_MODE>::kMN, B_MN = LoaderB<B_MODE>::kMN;
      const uint32_t idesc = make_idesc_tf32(bn, A_MN, B_MN);
      const uint32_t b_kgroup = (uint32_t)((bn + 31) >> 5) << 10;     // MN-major B: bytes per 8-k group
      int s = 0, ms = 0;                             // ms = i % n_main, kept incrementally
      uint32_t parity = 0;
      for (int i = 0; i < nkb; ++i) {
        mbar_wait(smem_u32(&sh->full[s]), parity);
        fence_proxy_async_smem();
        tc_fence_after();
        const uint32_t a_base = smem_base + s * stage_bytes;
        const uint32_t b_base = a_base + TC_A_BYTES;
        // K-major: advance 8 tf32 = 32 bytes inside the 128-byte swizzle row (+2 in the addr>>4 field);
        // MN-major: advance two 4-k groups of 512-byte atoms (A: 2 x 4 atoms = 4 KB; B: 2 x ceil(bn/32) atoms)
        const uint64_t adesc = A_MN ? make_smem_desc_mn(a_base, 512u, 2048u) : make_smem_desc(a_base);
        const uint64_t bdesc = B_MN ? make_smem_desc_mn(b_base, 512u, b_kgroup >> 1) : make_smem_desc(b_base);
        const uint64_t a_step = A_MN ? (uint64_t)(4096 >> 4) : 2ull, b_step = B_MN ? (uint64_t)(b_kgroup >> 4) : 2ull;
        const uint64_t lo_step = (uint64_t)(hi_bytes >> 4);   // residual tiles sit hi_bytes further (start-address field)
        // X3: both corrections accumulate in accumulator 0, hi*hi of K-block i in main accumulator 1 + i % n_main
        // (tmem_ld16_sum in offk_tc.cuh says why)
        const uint32_t acc_stride = ((uint32_t)bn + 31u) & ~31u;
        const uint32_t d_main = X3 ? tmem_d + (uint32_t)(1 + ms) * acc_stride : tmem_d;
        const bool main_started = X3 ? i >= n_main : i > 0;
        if (elect_one_sync()) {
#pragma unroll
          for (int j = 0; j < TC_BK / 8; ++j) {
            if (X3) {
              umma_tf32(tmem_d, adesc + lo_step + a_step * j, bdesc + b_step * j, idesc, (i > 0 || j > 0) ? 1u : 0u);
              umma_tf32(tmem_d, adesc + a_step * j, bdesc + lo_step + b_step * j, idesc, 1u);
            }
            umma_tf32(d_main, adesc + a_step * j, bdesc + b_step * j, idesc, (main_started || j > 0) ? 1u : 0u);
          }
          umma_commit(smem_u32(&sh->empty[s]));        // frees the smem slot when these MMAs retire
        }
        __syncwarp();
        if (++s == stages) { s = 0; parity ^= 1u; }
        if (++ms == n_main) ms = 0;
      }
      if (elect_one_sync()) umma_commit(smem_u32(&sh->accum_full));          // accumulator complete
    }
    __syncwarp();
  }

  // ================= epilogue (warps 0-7) =================
  if (warp < 8 && nkb > 0 && g.out_vec == 2) {
    // rows contiguous in memory (weight gradients): transposed float4 adds (offk_tc.cuh)
    mbar_wait(smem_u32(&sh->accum_full), 0u);
    tc_fence_after();
    epi_rows_contiguous(g, smem_base, tmem_d, X3 ? 1 + min(n_main, nkb) : 1, ((uint32_t)bn + 31u) & ~31u, bn, m0, n0, warp & 3,
                        warp >> 2, warp, lane, (g.split_k > 1) || g.atomic_out);
  } else if (warp < 8 && nkb > 0) {
    const int quad = warp & 3;                       // TMEM lane quadrant this warp may read
    const int m = m0 + quad * 32 + lane;
    const bool mvalid = m < g.M;
    // table entries first: they are in flight while the last MMAs retire
    EpiRow er = {0, 0, false};
    if (mvalid) er = epi_row(g, m);
    const bool atomic = (g.split_k > 1) || g.atomic_out;
    const bool vec = g.out_vec == 1 && !er.ones;
    // out_vec contract: column tables are contiguous (col[n] = col[0] + n)
    const int oc0 = __ldg(g.out_col);
    const int ac0 = g.addend ? (g.add_col ? __ldg(g.add_col) : oc0) : 0;
    mbar_wait(smem_u32(&sh->accum_full), 0u);
    tc_fence_after();
    const int nchunks = bn >> 4;
    for (int c = (warp >> 2); c < nchunks; c += 2) {  // warps 0-3 even 16-column chunks, 4-7 odd ones
      const int nb = n0 + c * 16;
      // Operands first (independent loads in flight), then the TMEM drain -- tcgen05.ld is .sync.aligned, so it is issued
      // by the whole warp outside any lane-divergent branch -- then math + stores.
      float4 gt[4], ad[4];
      int oc[16];
      const bool lane_vec = mvalid && vec;
      if (lane_vec) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int n = nb + 4 * j;
          ad[j] = f4zero(); gt[j] = make_float4(1.f, 1.f, 1.f, 1.f);
          if (n < g.N && !atomic) {
            if (g.gate && n >= g.gate_col0) gt[j] = ldg128(g.gate + (er.out + oc0 + n));
            if (g.addend) ad[j] = ldg128(g.addend + (er.add + ac0 + n));
          }
        }
      } else if (mvalid) {            // scalar path (weight gradients: out_col is a stride table)
#pragma unroll
        for (int j = 0; j < 16; ++j) oc[j] = (nb + j < g.N) ? __ldg(g.out_col + nb + j) : 0;
      }
      float v[16];
      tmem_ld16_sum(tmem_d + ((uint32_t)(quad * 32) << 16) + (uint32_t)(c * 16), X3 ? 1 + min(n_main, nkb) : 1,
                    ((uint32_t)bn + 31u) & ~31u, v);
      if (lane_vec) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int n = nb + 4 * j;
          if (n >= g.N) continue;
          float4 x = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          float* o = g.out + (er.out + oc0 + n);
          if (atomic) {
            asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(o), "f"(x.x), "f"(x.y), "f"(x.z), "f"(x.w) : "memory");
            continue;
          }
          const float4 bias4 = g.bias ? ldg128(g.bias + n) : f4zero();
          *reinterpret_cast<float4*>(o) = epi_act4(g, x, n, bias4, gt[j], ad[j], g.gate && n >= g.gate_col0);
        }
      } else if (mvalid) {
        if (atomic && !er.ones) {
#pragma unroll
          for (int j = 0; j < 16; ++j)
            if (nb + j < g.N) red_add_f32(g.out + (er.out + oc[j]), v[j]);
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int n = nb + j;
            if (n < g.N) epi_store(g, er, n, v[j], atomic);
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 8) {
    __syncwarp();
    tmem_dealloc(tmem_d, (uint32_t)tmem_cols);
  }
}

// ---------------------------------------------------------------------------- host
static int pick_bn(int N) {
  // one N tile when it fits a single UMMA (N <= 256, multiple of 16); otherwise the tile with least padding
  const int n16 = (N + 15) / 16 * 16;
  if (n16 <= 256) return n16;
  int best = 256, waste = 1 << 30;
  for (int bn = 256; bn >= 128; bn -= 16) {
    const int w = (N + bn - 1) / bn * bn - N;
    if (w < waste) { waste = w; best = bn; }
  }
  return best;
}

template <int A_MODE, int B_MODE, bool X3>
static int launch_tc_t(const offk_gemm_t& g, int bn, int stages, int kb_per, int tmem_cols, dim3 grid, size_t smem,
                       cudaStream_t st) {
  auto kern = gather_gemm_tc_kernel<A_MODE, B_MODE, X3>;
  const int la = stages - 1 < 3 ? stages - 1 : 3;      // X3: residual pass trails the cp.async issue front by `la` K-blocks
  int n_main = 1;
  if (X3) {   // (n_main + 1) accumulators of bn columns (32-column granules) in the allocated tensor memory, <= 4 mains
    n_main = tmem_cols / ((bn + 31) / 32 * 32) - 1;
    if (n_main > 4) n_main = 4;
    n_main = x3_main_accumulators(n_main, kb_per * (TC_BK / 8));
  }
  static bool attr_set = false;  // per instantiation
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return cuda_check(e, "cudaFuncSetAttribute(gather_gemm_tc)");
    attr_set = true;
  }
  cudaError_t e = launch_pdl(kern, grid, dim3(TC_THREADS), smem, st, g, bn, stages, kb_per, tmem_cols, la, n_main);
  if (e != cudaSuccess) return cuda_check(e, "gather_gemm_tc launch");
  return OFFK_LAUNCH_CHECK("gather_gemm_tc");
}

int launch_gemm_tc(const offk_gemm_t& g, cudaStream_t st, bool x3) {
  int bn = g.tile_n > 0 ? g.tile_n : pick_bn(g.N);
  if (bn % 16 != 0 || bn < 16 || bn > 256) return fail(OFFK_E_BADARG, "gather_gemm: bad N tile %d", bn);
  const int num_kb = (g.K + TC_BK - 1) / TC_BK;
  const int split = g.split_k > 1 ? g.split_k : 1;
  const int kb_per = (num_kb + split - 1) / split;
  const uint32_t stage_bytes = (TC_A_BYTES + (((bn + 31) >> 5) << 12)) * (x3 ? 2u : 1u);
  // two CTAs per SM: tiles of the same or of a concurrent kernel (another lane) co-reside; the 3xTF32 stages (twice the
  // bytes: residual tiles) of the wide tiles need the whole SM
  int budget = 108 * 1024;
  if (x3 && 3 * stage_bytes > (uint32_t)budget) budget = 216 * 1024;
  int stages = budget / (int)stage_bytes;
  if (stages < 2) stages = 2;
  if (stages > TC_MAX_STAGES) stages = TC_MAX_STAGES;
  if (stages > kb_per) stages = kb_per < 2 ? 2 : kb_per;
  const size_t smem = (size_t)stages * stage_bytes + sizeof(TcShared) + 1024;
  int tmem_cols = 32;
  while (tmem_cols < bn) tmem_cols <<= 1;
  if (x3) {   // room for the correction accumulator and up to 4 main ones: 256 columns while two CTAs share the SM, else 512
    const int cap = budget > 108 * 1024 ? 512 : 256, stride = (bn + 31) / 32 * 32;
    if (cap / stride < 2) return fail(OFFK_E_LIMIT, "gather_gemm: no room in tensor memory for the 3xTF32 accumulators (N tile %d)", bn);
    int want = (cap / stride > 5 ? 5 : cap / stride) * stride;
    tmem_cols = 32;
    while (tmem_cols < want) tmem_cols <<= 1;
    if (tmem_cols > cap) tmem_cols = cap;
  }
  dim3 grid((g.M + TC_BM - 1) / TC_BM, (g.N + bn - 1) / bn, (num_kb + kb_per - 1) / kb_per);
  if (grid.y > 65535 || grid.z > 65535) return fail(OFFK_E_LIMIT, "gather_gemm: grid too large");
#define OFFK_TC_CASE(AM, BM)                                                                        \
  if (g.a_mode == AM && g.b_mode == BM)                                                             \
    return x3 ? launch_tc_t<AM, BM, true>(g, bn, stages, kb_per, tmem_cols, grid, smem, st)         \
              : launch_tc_t<AM, BM, false>(g, bn, stages, kb_per, tmem_cols, grid, smem, st);
  OFFK_TC_CASE(OFFK_LOAD_VEC_K, OFFK_LOAD_VEC_K) OFFK_TC_CASE(OFFK_LOAD_VEC_K, OFFK_LOAD_VEC_ROW)
  OFFK_TC_CASE(OFFK_LOAD_VEC_ROW, OFFK_LOAD_VEC_K) OFFK_TC_CASE(OFFK_LOAD_VEC_ROW, OFFK_LOAD_VEC_ROW)
#undef OFFK_TC_CASE
  return fail(OFFK_E_BADARG, "gather_gemm: unsupported load modes %d/%d", g.a_mode, g.b_mode);
}

}  // namespace offk
