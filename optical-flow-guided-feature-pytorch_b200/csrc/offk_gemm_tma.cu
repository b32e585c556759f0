// TMA-fed tcgen05 GEMM (OFFK_PREC_TF32) for sm_100a: the dense contractions whose operands are regular enough for the
// Tensor Memory Accelerator -- every conv / FC of the OFF sub-network that works on channels-last tensors.
//
//   D[128 x BN] (fp32, TMEM) += A[128 x 32] (tf32, smem) * B[BN x 32]^T (tf32, smem)   per K-block
//
// Warp roles (320 threads):
//   warp 0     TMA producer: one elected lane waits for a free stage, posts mbarrier.arrive.expect_tx and issues
//              cp.async.bulk.tensor loads that land directly in the canonical SWIZZLE_128B shared-memory layouts:
//                A dense   : 2-D tile  {32 k, 128 rows}   of a row-major [M, lda] matrix (1x1 conv / FC input)
//                A im2col  : 4-D im2col {32 c, 128 pixels} of a channels-last [n, h, w, ctot] tensor at filter offset
//                            (q, r): the hardware walks the output pixels (stride, zero padding, image wrap) -- no index
//                            tables, no per-element predicates, one instruction per K-block
//                A nchw    : 3-D tiles {32 pixels, 32 c, 1 frame} of an NCHW [n, c, hw] tensor (the BN-Inception taps of
//                            the OFF units' fused 1x1 conv): pixels are contiguous, so the tile is the MN-major
//                            SWIZZLE_128B_BASE32B operand (tensor-map swizzle 128B_ATOM_32B) -- the NCHW -> channels-last
//                            conversion costs no instruction; M tiles never straddle a frame (OOB pixels zero-fill)
//                A nchw_t  : 3-D tile  {32 pixels, 128 c, 1 frame} of the same NCHW tensor with m = channel, k = pixel
//                            (weight gradient of the units' 1x1 conv): K-major; K-blocks are cut per frame
//                A im2col_t: up to four 4-D im2col atoms {32 c, 32 pixels} at the filter offsets of rows m = (r, q, c)
//                            with k = output pixel (weight gradient of a channels-last conv): MN-major
//                B dense   : 2-D tile  {32 k, BN rows}    of the [N, K] weight matrix (OHWI for KxK convs)
//                B dense_t : 2-D atoms {32 n, 32 k} of a row-major [K, ldb] matrix (the channels-last output gradient
//                            dY[pixel, cout] of a weight-gradient GEMM): MN-major
//              The all-ones A row of a weight-gradient GEMM (bias gradient, offk.h) cannot come from memory: it is
//              written into the landed tile by the MMA warp (generic proxy + fence.proxy.async), or into tensor memory by
//              the thread that owns the row when A goes there.  The K-block walk keeps (tap, channel block, pixel)
//              incrementally: no division in the loop.
//   warp 1     allocates TMEM; the warp waits on "full" (3xTF32: on "split") and one ELECTED lane (elect.sync -- under
//              `if (lane == 0)` every tcgen05.mma is wrapped in an ELECT / BRA.U.ANY loop, ~80 clocks apiece) issues
//              4 x tcgen05.mma (kind::tf32, M=128, N=BN, K=8) per stage -- 12 in the 3xTF32 mode --, tcgen05.commit's to the
//              stage's "empty" mbarrier and to "accum_full" after the last K-block
//   warps 2-9  main loop (3xTF32 only): the residual pass.  Each landed A tile is moved into TENSOR MEMORY as (hi, lo) column
//              pairs (tcgen05.st; the MMAs then take A from TMEM and read shared memory for B alone), or -- N tiles above 192,
//              where the accumulators fill TMEM -- gets a residual twin tile in shared memory; B_lo arrives by TMA from the
//              weights split once per step (offk_tf32_residual), or is written here for the weight-gradient kinds.
//              epilogue: tcgen05.ld the accumulator rows out of TMEM (warp w may touch TMEM lanes 32*(w%4)..+31; the 3xTF32
//              partial accumulators are summed in fp32 here) and leave through one of
//                * TMA tile stores (linear output rows, offk.h: out_ld): 32-column slabs staged in the SWIZZLE_128B box
//                  layout, cp.async.bulk.tensor stores, or cp.reduce...add for split-K partial sums
//                * 32-column chunks transposed through shared memory so that bias / ReLU / ReLU' gate / residual add and the
//                  float4 stores (red.global.add.v4 for split-K) touch whole 128-byte lines of the channels-last output
//                * the same transposition the other way round for weight gradients (out_vec = 2: dW[n][m], 4 rows per lane)
// One output tile per CTA; two CTAs co-reside per SM in the tf32 mode so one CTA's epilogue overlaps the other's main loop
// (the 3xTF32 stages and TMEM budget take the whole SM).  tools/timeline.py + -DOFFK_TIMELINE stamp every phase per CTA.
#include <cuda.h>
#include "offk_tc.cuh"

namespace offk {

constexpr int TM_THREADS = 320;          // TMA warp, MMA warp, 8 epilogue warps
constexpr int TM_EPI_PITCH = 36;          // floats per row of the epilogue staging tile (32 columns + 4 padding)

struct TmGeom {        // what the producer needs to turn (tile, K-block) into TMA coordinates
  int a_kind;
  int a_coff;          // first channel of the A operand inside its buffer (im2col)
  int cblocks;         // cin / 32 (im2col)
  int kw;              // filter width (im2col)
  int hout, wout, stride, pad, pad_w;   // pad = top rows, pad_w = left columns (equal unless OFFK_TGEMM_FREE_GEOM)
  int hw, tiles_per_img;   // nchw: pixels per frame, M tiles per frame
  int kb_per_img;          // nchw_t: K-blocks per frame (ceil(hw / 32))
  int kw_rows;             // im2col_t: kh*kw*cin = number of real A rows (the ones row follows)
};

__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(tm), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, int c2, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(dst),
      "l"(tm), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_im2col_4d(uint32_t dst, const CUtensorMap* tm, int c, int w, int h, int n,
                                                   int woff, int hoff, uint32_t bar) {
  const unsigned short wo = (unsigned short)woff, ho = (unsigned short)hoff;
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.im2col.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2], "
      "{%7, %8};" ::"r"(dst),
      "l"(tm), "r"(bar), "r"(c), "r"(w), "r"(h), "r"(n), "h"(wo), "h"(ho)
      : "memory");
}
// shared -> global tile stores / float adds through the TMA (bulk async-group completion)
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* tm, uint32_t src, int c0, int c1, bool add) {
  if (add)
    asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];" ::"l"(tm), "r"(src),
                 "r"(c0), "r"(c1)
                 : "memory");
  else
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%2, %3}], [%1];" ::"l"(tm), "r"(src), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* tm, uint32_t src, int c0, int c1, int c2, bool add) {
  if (add)
    asm volatile("cp.reduce.async.bulk.tensor.3d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(tm), "r"(src),
                 "r"(c0), "r"(c1), "r"(c2)
                 : "memory");
  else
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(tm), "r"(src), "r"(c0),
                 "r"(c1), "r"(c2)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tm) : "memory");
}

// Diagnostics build only (-DOFFK_TIMELINE, tools/timeline.py): per-CTA clock64 stamps of the kernel's phases.
#ifdef OFFK_TIMELINE
constexpr int TL_MAX_CTAS = 8192, TL_SLOTS = 32;
__device__ long long tl_buf[TL_MAX_CTAS * TL_SLOTS];
#define TL_STAMP(slot)                                                                                      \
  do {                                                                                                      \
    const int cta_ = (blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;                        \
    if (cta_ < TL_MAX_CTAS) tl_buf[cta_ * TL_SLOTS + (slot)] = clock64();                                   \
  } while (0)
#else
#define TL_STAMP(slot) do { } while (0)
#endif

struct TmShared {
  uint64_t full[TC_MAX_STAGES];
  uint64_t empty[TC_MAX_STAGES];
  uint64_t accum_full;
  uint64_t split[TC_MAX_STAGES];   // X3: the residual ("lo") tiles of the stage are written (256 epilogue threads)
  uint32_t tmem_base;
  uint32_t last_flag;              // split-K finisher: 1 in the CTA that arrived last on the tile's counter
  float bias[256];                 // the tile's bias values (vector epilogue)
};

// Final value of 4 consecutive elements (one accumulator row, columns n..n+3): the epilogue of offk.h (epi_act4), then the
// optional second output.  out_base / aux_base: element offsets of the row in `out` / `aux_out` (column 0).
__device__ __forceinline__ float4 epi_final4(const offk_gemm_t& g, float4 v, int n, const float4& bias4, const float4& t,
                                             const float4& ad, bool gated, int out_base, int aux_base) {
  v = epi_act4(g, v, n, bias4, t, ad, gated);
  if (g.aux_out) {
    float4 a = v;
    if (g.aux_addend) {
      const float4 x = ldg128(g.aux_addend + (out_base + n));
      a.x += x.x; a.y += x.y; a.z += x.z; a.w += x.w;
    }
    *reinterpret_cast<float4*>(g.aux_out + (aux_base + n)) = f4relu(a);
  }
  return v;
}

// Split-K finisher (offk.h: finish_counter), called by the 256 epilogue threads of every split CTA after their partial tile
// went out as red.global.add: the last CTA to arrive on the tile's counter re-reads the summed tile and applies the epilogue
// in place.  Kept out of line: it runs once per output tile, and its registers must not weigh on the main kernel.
// release: this thread's reds, fence, CTA barrier, counter; acquire: counter, barrier, fence, .cg loads.
__device__ __noinline__ void splitk_finish(const offk_gemm_t& g, uint32_t* flag_smem, int etid, int m0, int m_lim, int n0, int bn) {
  __threadfence();
  asm volatile("bar.sync 1, 256;" ::: "memory");
  volatile uint32_t* flag = flag_smem;
  if (etid == 0) {
    int* ctr = g.finish_counter + (blockIdx.y * gridDim.x + blockIdx.x);
    const int prev = atomicAdd(ctr, 1);
    const int last = prev == (int)gridDim.z - 1;
    if (last) *ctr = 0;                                    // ready for the next launch / graph replay
    *flag = (uint32_t)last;
  }
  asm volatile("bar.sync 1, 256;" ::: "memory");
  if (!*flag) return;
  __threadfence();
  const int oc0 = __ldg(g.out_col);
  const int ac0 = g.addend ? (g.add_col ? __ldg(g.add_col) : oc0) : 0;
  const int c4n = bn >> 2;                                 // float4 columns of the tile
  // thread -> (row, float4 column): consecutive threads walk a row (coalesced), 256 threads cover 256 / c4n rows per pass
  for (int i = etid; i < TC_BM * c4n; i += 256) {
    const int row = i / c4n, n = n0 + (i - row * c4n) * 4, m = m0 + row;
    if (m >= m_lim || n >= g.N) continue;
    const EpiRow er = epi_row(g, m);
    const int aux_base = g.aux_out ? (g.aux_row ? __ldg(g.aux_row + m) : er.out) : 0;
    const bool gated = g.gate && n >= g.gate_col0;
    float* o = g.out + (er.out + oc0 + n);
    const float4 v = __ldcg(reinterpret_cast<const float4*>(o));
    const float4 bias4 = g.bias ? ldg128(g.bias + n) : f4zero();
    const float4 t = gated ? ldg128(g.gate + (er.out + oc0 + n)) : make_float4(1.f, 1.f, 1.f, 1.f);
    const float4 ad4 = g.addend ? ldg128(g.addend + (er.add + ac0 + n)) : f4zero();
    *reinterpret_cast<float4*>(o) = epi_final4(g, v, n, bias4, t, ad4, gated, er.out + oc0, aux_base);
  }
}

// X3 = OFFK_PREC_TF32X3: the epilogue warps, otherwise idle during the main loop, turn each landed tile into (hi, lo) --
// A into tensor memory (a_tmem > 0: stage = [A | B | B_lo]) or into a twin tile (stage = [A | B | A_lo | B_lo]) -- and the
// MMA warp issues three MMAs per K = 8 step (offk_tc.cuh: tf32_lo, tmem_ld16_sum).
template <int A_KIND, int B_KIND, bool X3>
// (launch bounds: 3xTF32 runs one CTA per SM anyway -- stage size -- and needs the registers for the five partial
// accumulators of a drained chunk)
__global__ void __launch_bounds__(TM_THREADS, X3 ? 1 : 2)
tma_gemm_kernel(const __grid_constant__ CUtensorMap tma, const __grid_constant__ CUtensorMap tmb, const __grid_constant__ CUtensorMap tmc,
                const __grid_constant__ offk_gemm_t g, const TmGeom geo, int bn, int stages, int kb_per_split, int tmem_cols, int n_main,
                int bk, int b_presplit, int a_tmem, int c_mode) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  constexpr bool A_MN = (A_KIND == OFFK_TMA_A_NCHW || A_KIND == OFFK_TMA_A_IM2COL_T);   // MN-major operand tiles
  constexpr bool B_MN = (B_KIND == OFFK_TMA_B_DENSE_T);
  // K-block depth: 32 (one 128-byte swizzle row) whenever an operand is K-major; `bk` (32 / 64 / 128 output pixels) for the
  // channels-last weight gradient, whose operands are both MN-major stacks of {32 m|n x 4 k} atoms along k -- deeper
  // K-blocks mean fewer, larger TMA boxes per byte (a 32-pixel im2col box is 4 KB: the TMA unit, not L2, was the limit)
  const uint32_t atom_bytes = (uint32_t)bk * 128u;              // one {32 m|n x bk k} MN-major stack
  const uint32_t a_bytes = A_KIND == OFFK_TMA_A_IM2COL_T ? 4u * atom_bytes : (uint32_t)TC_A_BYTES;
  const uint32_t b_bytes = B_MN ? (((uint32_t)bn + 31u) >> 5) * atom_bytes : (uint32_t)bn * 128u;
  const uint32_t hi_bytes = a_bytes + b_bytes;                  // one landed [A | B] pair
  const uint32_t blo_bytes = (X3 && !B_MN && b_presplit) ? b_bytes : 0u;   // residual B tile delivered by TMA as well
  // X3 with the A operand in tensor memory (a_tmem): the epilogue warps move each landed A tile into TMEM as (hi, lo)
  // column pairs instead of writing a residual tile next to it; the three MMAs of a K = 8 step then read shared memory
  // for B only.  Stage = [A | B | B_lo]; TMEM = [accumulators | stage 0: A_hi, A_lo | stage 1: ... ].
  const bool atm = X3 && a_tmem != 0;
  const uint32_t lo_off = atm ? b_bytes : hi_bytes;             // residual tile = its hi tile + lo_off
  const uint32_t stage_bytes = X3 ? (atm ? hi_bytes + b_bytes : 2u * hi_bytes) : hi_bytes;
  const uint32_t a_cols = A_KIND == OFFK_TMA_A_IM2COL_T ? (uint32_t)bk : (uint32_t)TC_BK;   // K-block depth = TMEM columns of A_hi
  // barriers etc. sit behind the pipeline stages -- or behind the epilogue's staging buffers where those are larger
  const uint32_t epi_bytes = c_mode ? 3u * TC_BM * 128u : 2u * TC_BM * TM_EPI_PITCH * 4u;
  const uint32_t pipe_bytes = max((uint32_t)stages * stage_bytes, epi_bytes);
  TmShared* sh = reinterpret_cast<TmShared*>(smem_raw + (smem_base - smem_u32(smem_raw)) + pipe_bytes);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) TL_STAMP(0);                                     // kernel entry
  int m0 = blockIdx.x * TC_BM, m_lim = g.M;
  int img_t = 0, pix0 = 0;
  if (A_KIND == OFFK_TMA_A_NCHW) {                               // M tiles are cut per frame
    img_t = blockIdx.x / geo.tiles_per_img;
    pix0 = (blockIdx.x - img_t * geo.tiles_per_img) * TC_BM;
    m0 = img_t * geo.hw + pix0;
    m_lim = min(g.M, (img_t + 1) * geo.hw);
  }
  const int n0 = blockIdx.y * bn;
  const int num_kb_total = A_KIND == OFFK_TMA_A_NCHW_T ? (g.K / geo.hw) * geo.kb_per_img : (g.K + bk - 1) / bk;
  const int kb_begin = blockIdx.z * kb_per_split;
  const int kb_end = min(num_kb_total, kb_begin + kb_per_split);
  const int nkb = kb_end - kb_begin;

  if (tid == 0) {
    for (int s = 0; s < stages; ++s) {
      mbar_init(smem_u32(&sh->full[s]), 1);
      mbar_init(smem_u32(&sh->empty[s]), 1);
      if (X3) mbar_init(smem_u32(&sh->split[s]), TM_THREADS - 64);
    }
    mbar_init(smem_u32(&sh->accum_full), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    tma_prefetch_desc(&tma);
    tma_prefetch_desc(&tmb);
    if (c_mode) tma_prefetch_desc(&tmc);
  }
  if (warp == 1) tmem_alloc(smem_u32(&sh->tmem_base), (uint32_t)tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_d = sh->tmem_base;
  // Programmatic dependent launch: everything above (barrier init, TMEM allocation, tensor-map prefetch) may overlap
  // the tail of the previous kernel in the stream; nothing below runs before that kernel's memory is visible.  The
  // next kernel may begin ITS prologue once every CTA of this grid got past the wait.  (No-ops without the attribute.)
  if (tid == 0) TL_STAMP(1);                                     // prologue done
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (tid == 0) TL_STAMP(2);                                     // predecessor's memory visible

  if (warp == 0) {
    {
      // ================= TMA producer (converged warp, one elected lane issues: see elect_one_sync) =================
      int w0 = 0, h0 = 0, img0 = 0;
      if (A_KIND == OFFK_TMA_A_IM2COL) {
        const int hw = geo.hout * geo.wout;
        img0 = m0 / hw;
        const int rem = m0 - img0 * hw;
        const int oy = rem / geo.wout, ox = rem - oy * geo.wout;
        w0 = ox * geo.stride - geo.pad_w;
        h0 = oy * geo.stride - geo.pad;
      }
      // K-block walk without divisions in the loop (they cost the issuing lane ~100 clocks each: 1800 clocks per K-block
      // of the 7x7 weight gradient, profiles/timeline_fp32_r02r): the position of K-block kb_begin is decomposed once,
      // then advanced incrementally.
      int it_cb = 0, it_q = 0, it_r = 0;                         // im2col: channel block, filter column, filter row
      int it_img = 0, it_pb = 0;                                 // nchw_t: frame, pixel block inside the frame
      int it_ox = 0, it_oy = 0, it_im = 0;                       // im2col_t: first output pixel of the K-block
      int at_q[TC_BM / 32], at_r[TC_BM / 32], at_c[TC_BM / 32];  // im2col_t: the four row atoms' (q, r, first channel)
      if (A_KIND == OFFK_TMA_A_IM2COL) {
        const int tap = kb_begin / geo.cblocks;
        it_cb = kb_begin - tap * geo.cblocks;
        it_r = tap / geo.kw;
        it_q = tap - it_r * geo.kw;
      }
      if (A_KIND == OFFK_TMA_A_NCHW_T) {
        it_img = kb_begin / geo.kb_per_img;
        it_pb = kb_begin - it_img * geo.kb_per_img;
      }
      if (A_KIND == OFFK_TMA_A_IM2COL_T) {
        const int hwo = geo.hout * geo.wout;
        const int p0 = kb_begin * bk;
        it_im = p0 / hwo;
        const int rem = p0 - it_im * hwo;
        it_oy = rem / geo.wout;
        it_ox = rem - it_oy * geo.wout;
#pragma unroll
        for (int a = 0; a < TC_BM / 32; ++a) {
          const int at = (m0 >> 5) + a;
          const int tap = at / geo.cblocks, cb = at - tap * geo.cblocks;
          at_r[a] = tap / geo.kw;
          at_q[a] = tap - at_r[a] * geo.kw;
          at_c[a] = geo.a_coff + cb * TC_BK;
        }
      }
      int s = 0;
      uint32_t parity = 1;                                       // empty-barrier parity of the current round
      for (int i = 0; i < nkb; ++i) {
        const int kb = kb_begin + i;
        mbar_wait(smem_u32(&sh->empty[s]), parity);              // slot free (first round passes at once)
        if (i == 8 && lane == 0) TL_STAMP(16);
        if (i == 9 && lane == 0) TL_STAMP(22);
        if (elect_one_sync()) {
        const uint32_t full = smem_u32(&sh->full[s]);
        const uint32_t a_dst = smem_base + s * stage_bytes;
        const uint32_t b_dst = a_dst + a_bytes;
        int b_row0 = kb * bk;                                    // dense_t: first k (pixel) row of this K-block
        if (A_KIND == OFFK_TMA_A_NCHW) {
          // four 4 KB atoms {32 pixels x 32 channels}; atoms wholly past the frame end are skipped (their
          // accumulator rows are never stored)
          const int n_at = min(TC_BM / 32, (geo.hw - pix0 + 31) >> 5);
          mbar_arrive_expect_tx(full, (uint32_t)n_at * 4096u + b_bytes + blo_bytes);
          for (int a = 0; a < n_at; ++a) tma_load_3d(a_dst + a * 4096, &tma, pix0 + 32 * a, kb * TC_BK, img_t, full);
        } else if (A_KIND == OFFK_TMA_A_NCHW_T) {
          // K-block = 32 pixels of ONE frame (pixels past the frame end zero-fill, so whatever rows of dY they meet
          // contribute nothing); rows = 128 channels (channels >= cin zero-fill; the ones row is patched in)
          const int img = it_img, pb = it_pb;
          b_row0 = img * geo.hw + pb * TC_BK;
          mbar_arrive_expect_tx(full, hi_bytes + blo_bytes);
          tma_load_3d(a_dst, &tma, pb * TC_BK, m0, img, full);
        } else if (A_KIND == OFFK_TMA_A_IM2COL_T) {
          // rows m = (r, q, c): each 32-row atom is one {32 channels x 32 output pixels} im2col box at its own (q, r)
          const int at0 = m0 >> 5;
          const int n_at = max(0, min(TC_BM / 32, (geo.kw_rows >> 5) - at0));
          mbar_arrive_expect_tx(full, (uint32_t)n_at * atom_bytes + b_bytes + blo_bytes);
          const int wb = it_ox * geo.stride - geo.pad_w, hb = it_oy * geo.stride - geo.pad;
#pragma unroll
          for (int a = 0; a < TC_BM / 32; ++a)
            if (a < n_at) tma_load_im2col_4d(a_dst + a * atom_bytes, &tma, at_c[a], wb, hb, it_im, at_q[a], at_r[a], full);
        } else if (A_KIND == OFFK_TMA_A_DENSE) {
          mbar_arrive_expect_tx(full, hi_bytes + blo_bytes);
          tma_load_2d(a_dst, &tma, kb * TC_BK, m0, full);
        } else {
          mbar_arrive_expect_tx(full, hi_bytes + blo_bytes);
          tma_load_im2col_4d(a_dst, &tma, geo.a_coff + it_cb * TC_BK, w0, h0, img0, it_q, it_r, full);
        }
        if (B_MN) {
          const int n_bat = (bn + 31) >> 5;
          for (int a = 0; a < n_bat; ++a) tma_load_2d(b_dst + a * atom_bytes, &tmb, n0 + 32 * a, b_row0, full);
        } else if (X3 && b_presplit) {
          // weights split ahead of time (offk.h: b_lo_delta): the residual matrix is plane 1 of a 3-D tensor map and lands
          // straight in the stage's B_lo slot -- no shared-memory pass over the weight tile
          tma_load_3d(b_dst, &tmb, kb * TC_BK, n0, 0, full);
          tma_load_3d(b_dst + lo_off, &tmb, kb * TC_BK, n0, 1, full);
        } else {
          tma_load_2d(b_dst, &tmb, kb * TC_BK, n0, full);
        }
        }
        __syncwarp();
        if (A_KIND == OFFK_TMA_A_IM2COL) {
          if (++it_cb == geo.cblocks) { it_cb = 0; if (++it_q == geo.kw) { it_q = 0; ++it_r; } }
        }
        if (A_KIND == OFFK_TMA_A_NCHW_T) {
          if (++it_pb == geo.kb_per_img) { it_pb = 0; ++it_img; }
        }
        if (A_KIND == OFFK_TMA_A_IM2COL_T) {
          it_ox += bk;
          while (it_ox >= geo.wout) { it_ox -= geo.wout; if (++it_oy == geo.hout) { it_oy = 0; ++it_im; } }
        }
        if (i == 8 && lane == 0) TL_STAMP(17);                   // steady-state K-block: loads issued
        if (++s == stages) { s = 0; parity ^= 1u; }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ================= MMA issuer (one elected lane; the whole warp when it must patch the ones row) =================
    // K-major: +32 bytes inside the 128-byte swizzle row per K = 8.  MN-major: 512-byte atoms of {32 m|n x 4 k}; a
    // TMA box stacks the 8 k-groups of one 32-wide atom (SBO 512), the atoms along m|n follow at 4 KB (LBO);
    // K = 8 advances two k-groups.
    const uint32_t idesc = make_idesc_tf32(bn, A_MN && !atm, B_MN);
    const uint32_t acc_cols = (((uint32_t)bn + 31u) & ~31u) * (uint32_t)(1 + n_main);   // a_tmem: A slots follow the accumulators
    const uint64_t a_step = A_MN ? (uint64_t)(1024 >> 4) : 2ull, b_step = B_MN ? (uint64_t)(1024 >> 4) : 2ull;
    constexpr bool kOnes = (A_KIND == OFFK_TMA_A_NCHW_T || A_KIND == OFFK_TMA_A_IM2COL_T);
    const int ones_loc = g.a_ones_row - m0;                       // row of this tile that must read all-ones
    const bool patch = kOnes && ones_loc >= 0 && ones_loc < TC_BM && !atm;   // a_tmem: patched on the way into TMEM
    {                                                             // the whole warp stays converged; one elected lane issues
      int s = 0, ts = 0, ms = 0;                                  // ts / ms: i % a_tmem / i % n_main, kept incrementally (an
      uint32_t parity = 0;                                        // integer modulo costs the issuing lane ~100 clocks per K-block)
      for (int i = 0; i < nkb; ++i) {
        mbar_wait(smem_u32(X3 ? &sh->split[s] : &sh->full[s]), parity);
        tc_fence_after();
        if (i == 0 && lane == 0) TL_STAMP(3);                    // first K-block ready for the tensor core
        if (i == 8 && lane == 0) TL_STAMP(20);
        if (i == 9 && lane == 0) TL_STAMP(24);
        const uint32_t a_base = smem_base + s * stage_bytes;
        if (patch) {
          // lane = k inside the K-block; 1 for real pixels, 0 past the end (of the frame: nchw_t; of K: im2col_t)
          const int kb = kb_begin + i;
          bool real;
          uint32_t off;
          if (A_KIND == OFFK_TMA_A_NCHW_T) {
            const int pb = kb - (kb / geo.kb_per_img) * geo.kb_per_img;
            real = pb * TC_BK + lane < geo.hw;
            off = swz(ones_loc, lane >> 2) + (uint32_t)(lane & 3) * 4u;
          } else {
            real = kb * bk + lane < g.K;
            const int ma = ones_loc >> 5, mi = ones_loc & 31, kl = lane & 3;
            off = (uint32_t)(ma * atom_bytes + (lane >> 2) * 512 + kl * 128 + ((((mi >> 3) ^ kl) << 5) | ((mi & 7) << 2)));
            for (int k2 = 32; k2 < bk; k2 += 32) {               // deeper K-blocks: the same row, 32 k further per pass
              const uint32_t o2 = off + (uint32_t)(k2 >> 2) * 512u;
              sts32(a_base + o2, kb * bk + k2 + lane < g.K ? 1.f : 0.f);
              if (X3) sts32(a_base + hi_bytes + o2, 0.f);
            }
          }
          sts32(a_base + off, real ? 1.f : 0.f);
          if (X3) sts32(a_base + hi_bytes + off, 0.f);           // 1 and 0 are exact in tf32: no residual
          fence_proxy_async_smem();
          __syncwarp();
        }
        if (elect_one_sync()) {
          const uint64_t adesc = A_MN ? make_smem_desc_mn(a_base, A_KIND == OFFK_TMA_A_IM2COL_T ? atom_bytes : 4096u, 512u) : make_smem_desc(a_base);
          const uint64_t bdesc = B_MN ? make_smem_desc_mn(a_base + a_bytes, atom_bytes, 512u) : make_smem_desc(a_base + a_bytes);
          const int ksteps = (A_KIND == OFFK_TMA_A_IM2COL_T ? bk : TC_BK) / 8;
          const uint64_t lo_step = (uint64_t)(lo_off >> 4);      // residual tiles sit lo_off further (start-address field)
          // X3: both corrections accumulate in accumulator 0, hi*hi of K-block i in main accumulator 1 + i % n_main
          const uint32_t acc_stride = ((uint32_t)bn + 31u) & ~31u;
          const uint32_t d_main = X3 ? tmem_d + (uint32_t)(1 + ms) * acc_stride : tmem_d;
          const uint32_t d_corr = tmem_d;
          const bool main_started = X3 ? i >= n_main : i > 0;
          if (atm) {
            const uint32_t a_hi = tmem_d + acc_cols + (uint32_t)ts * 2u * a_cols, a_lo = a_hi + a_cols;
#pragma unroll 4
            for (int j = 0; j < ksteps; ++j) {
              umma_tf32_ta(d_corr, a_lo + 8u * j, bdesc + b_step * j, idesc, (i > 0 || j > 0) ? 1u : 0u);
              umma_tf32_ta(d_corr, a_hi + 8u * j, bdesc + lo_step + b_step * j, idesc, 1u);
              umma_tf32_ta(d_main, a_hi + 8u * j, bdesc + b_step * j, idesc, (main_started || j > 0) ? 1u : 0u);
            }
          } else
#pragma unroll 4
          for (int j = 0; j < ksteps; ++j) {
            if (X3) {
              umma_tf32(d_corr, adesc + lo_step + a_step * j, bdesc + b_step * j, idesc, (i > 0 || j > 0) ? 1u : 0u);
              umma_tf32(d_corr, adesc + a_step * j, bdesc + lo_step + b_step * j, idesc, 1u);
            }
            umma_tf32(d_main, adesc + a_step * j, bdesc + b_step * j, idesc, (main_started || j > 0) ? 1u : 0u);
          }
          umma_commit(smem_u32(&sh->empty[s]));                  // frees the smem slot when these MMAs retire
          if (i == 8) TL_STAMP(21);
          if (i == 9) TL_STAMP(25);
        }
        __syncwarp();
        if (++s == stages) { s = 0; parity ^= 1u; }
        if (++ts == a_tmem) ts = 0;
        if (++ms == n_main) ms = 0;
      }
      if (elect_one_sync()) umma_commit(smem_u32(&sh->accum_full));     // accumulator complete
      if (lane == 0) TL_STAMP(4);                                // last MMA issued
    }
    __syncwarp();
  } else if (nkb > 0) {
    // ================= epilogue (warps 2-9) =================
    const int ew = warp - 2;                                     // 0..7
    const int quad = warp & 3;                                   // TMEM lane quadrant this warp may read
    const int half = ew >> 2;                                    // which 16 columns of a 32-column chunk
    const bool atomic = (g.split_k > 1) || g.atomic_out;
    // accumulators to add up in the epilogue (X3: the correction accumulator + the main ones that received a K-block)
    const int n_acc = X3 ? 1 + min(n_main, nkb) : 1;
    const uint32_t acc_stride = ((uint32_t)bn + 31u) & ~31u;
    // X3 main-loop duty of these 256 threads: residual tiles.  Stage s = [A | B | A_lo | B_lo]; the first half is what
    // the TMA delivered, the second half is written here, element for element at the same swizzled offset.
    auto split_loop = [&]() {
      if (!X3) return;
      const uint32_t e16 = (uint32_t)(tid - 64) * 16u;
      const uint32_t acc_cols = acc_stride * (uint32_t)(1 + n_main);
      constexpr bool kOnes = (A_KIND == OFFK_TMA_A_NCHW_T || A_KIND == OFFK_TMA_A_IM2COL_T);
      const int row = quad * 32 + lane;                          // a_tmem: the A row (= TMEM lane) this thread moves
      const bool ones_row = kOnes && row == g.a_ones_row - m0;
      int s = 0;
      uint32_t parity = 0;
      int fs = 0, ts = 0;                                        // a_tmem: slot of K-block i; stage / parity of K-block
      uint32_t fparity = 0;                                      // i - a_tmem, whose MMAs must retire before the slot is rewritten
      for (int i = 0; i < nkb; ++i) {
        mbar_wait(smem_u32(&sh->full[s]), parity);
        if (i == 0 && tid == 64) TL_STAMP(13);                   // first K-block landed
        if (i == 8 && tid == 64) TL_STAMP(18);
        if (i == 9 && tid == 64) TL_STAMP(23);
        const uint32_t base = smem_base + s * stage_bytes;
        if (atm) {
          // A tile -> tensor memory: 16 consecutive k of this thread's row per pass (the two warps of a lane quadrant
          // take alternate 16-column groups), hi = the 19 bits the tensor core reads, lo = rn_tf32(x - hi)
          // a_tmem = number of (A_hi, A_lo) column pairs: fewer than pipeline stages when the accumulators need the
          // room -- the landed tiles then wait in shared memory for the MMAs of K-block i - a_tmem (their commit on
          // that stage's "empty" barrier) before they may move in
          if (a_tmem < stages && i >= a_tmem) {                  // (as many slots as stages: the producer waited already)
            mbar_wait(smem_u32(&sh->empty[fs]), fparity);
            tc_fence_after();
            if (++fs == stages) { fs = 0; fparity ^= 1u; }
          }
          const uint32_t t_hi = tmem_d + ((uint32_t)(quad * 32) << 16) + acc_cols + (uint32_t)ts * 2u * a_cols;
          if (++ts == a_tmem) ts = 0;
          const int kb = kb_begin + i;
          for (uint32_t kk = (uint32_t)half * 16u; kk < a_cols; kk += 32u) {
            float x[16];
            if (A_MN) {
              const uint32_t abytes = A_KIND == OFFK_TMA_A_IM2COL_T ? atom_bytes : 4096u;
              const uint32_t rb = base + (uint32_t)quad * abytes + (uint32_t)((lane & 7) << 2);
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                const uint32_t k = kk + j;
                x[j] = lds32(rb + k * 128u + ((((uint32_t)(lane >> 3)) ^ (k & 3u)) << 5));
              }
            } else {
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float4 v = lds128(base + swz(row, (int)(kk >> 2) + j));
                x[4 * j] = v.x; x[4 * j + 1] = v.y; x[4 * j + 2] = v.z; x[4 * j + 3] = v.w;
              }
            }
            if (ones_row) {                                      // bias-gradient row: 1 for real k, 0 past the end
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                bool real;
                if (A_KIND == OFFK_TMA_A_NCHW_T) real = (kb - (kb / geo.kb_per_img) * geo.kb_per_img) * TC_BK + (int)kk + j < geo.hw;
                else real = kb * bk + (int)kk + j < g.K;
                x[j] = real ? 1.f : 0.f;
              }
            }
            uint32_t hi[16], lo[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              hi[j] = __float_as_uint(x[j]) & 0xFFFFE000u;
              lo[j] = __float_as_uint(tf32_lo(x[j]));
            }
            tmem_st16(t_hi + kk, hi);
            tmem_st16(t_hi + a_cols + kk, lo);
          }
          if (!blo_bytes) {                                      // B not split ahead of time (weight-gradient kinds)
#pragma unroll 4
            for (uint32_t off = e16; off < b_bytes; off += (TM_THREADS - 64) * 16u) split_chunk(base + a_bytes + off, lo_off);
            fence_proxy_async_smem();
          }
          tmem_st_wait();
          tc_fence_before();
        } else {
          const uint32_t split_bytes = blo_bytes ? a_bytes : hi_bytes;     // pre-split weights: only the A tile needs the pass
#pragma unroll 4
          for (uint32_t off = e16; off < split_bytes; off += (TM_THREADS - 64) * 16u) split_chunk(base + off, hi_bytes);
          fence_proxy_async_smem();                              // generic-proxy writes -> visible to tcgen05.mma
        }
        mbar_arrive(smem_u32(&sh->split[s]));
        if (i == 0 && tid == 64) TL_STAMP(14);                   // ... and split
        if (i == 8 && tid == 64) TL_STAMP(19);
        if (++s == stages) { s = 0; parity ^= 1u; }
      }
    };
    if (g.out_vec == 1 && c_mode != 0) {
      // Linear output rows (offk.h: out_ld): 32-column slabs of the tile go to shared memory in the SWIZZLE_128B box
      // layout (row r at r * 128 bytes, 16-byte chunk j at j ^ (r & 7)) and leave as TMA tile stores -- or float adds
      // for split-K partial sums -- which clip at the matrix / frame edge.  Three slabs rotate: the store of slab c - 2
      // has released its buffer (wait_group.read) before anyone passed the barrier of slab c - 1.  One accumulator row per
      // thread: bias and ReLU only (host: no gate, addend, finisher or second output on this path).
      if (g.bias && !atomic)
        for (int i = tid - 64; i < bn; i += TM_THREADS - 64) sh->bias[i] = n0 + i < g.N ? __ldg(g.bias + n0 + i) : 0.f;
      asm volatile("bar.sync 1, 256;" ::: "memory");             // bias values are read before the first slab barrier
      split_loop();
      if (tid == 64) TL_STAMP(5);
      mbar_wait(smem_u32(&sh->accum_full), 0u);
      tc_fence_after();
      if (tid == 64) TL_STAMP(6);
      const int trow = quad * 32 + lane;
      const int nchunks = bn >> 5;                               // host: bn % 32 == 0 on this path
      int slab = 0;
      for (int c = 0; c < nchunks; ++c) {
        const uint32_t buf = smem_base + (uint32_t)slab * (TC_BM * 128);
        float v[16];
        tmem_ld16_sum(tmem_d + ((uint32_t)(quad * 32) << 16) + (uint32_t)(c * 32 + half * 16), n_acc, acc_stride, v);
        const int nl = c * 32 + half * 16;                       // first of this thread's 16 columns inside the tile
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
          float4 x = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
          if (!atomic) {
            if (g.bias) {
              const float4 b = *reinterpret_cast<const float4*>(&sh->bias[nl + j]);
              x.x += b.x; x.y += b.y; x.z += b.z; x.w += b.w;
            }
            if (n0 + nl + j < g.relu_pre_cols || g.relu_post) x = f4relu(x);
          }
          sts128(buf + (uint32_t)trow * 128u + (uint32_t)((((half * 4 + (j >> 2))) ^ (trow & 7)) << 4), x.x, x.y, x.z, x.w);
        }
        fence_proxy_async_smem();                                // generic-proxy writes -> visible to the TMA
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (warp == 2 && elect_one_sync()) {
          if (c_mode == 2) tma_store_3d(&tmc, buf, n0 + c * 32, pix0, img_t, atomic);
          else tma_store_2d(&tmc, buf, n0 + c * 32, m0, atomic);
          tma_store_commit();
          tma_store_wait_read<1>();                              // slab c - 1 may still be read; slab c - 2 is free
        }
        if (++slab == 3) slab = 0;
      }
      if (warp == 2 && elect_one_sync()) tma_store_wait_read<0>();   // shared memory must outlive the reads
      if (tid == 64) TL_STAMP(12);
    } else if (g.out_vec == 1) {
      // Transposed through shared memory (the pipeline stages are idle once accum_full fired) so that bias / gate /
      // residual loads and the stores are row-contiguous: 8 lanes x 16 bytes = one 128-byte line per output row.
      // Staging tile: 128 rows x 32 columns, row pitch 36 floats (conflict-free 128-bit accesses), double-buffered.
      const uint32_t stg0 = smem_base;
      const int trow = quad * 32 + lane;                         // accumulator row this thread drains
      const int rsub = lane >> 3, cq = lane & 7;                 // read-back: 4 rows per warp pass, 8 float4 per row
      const int nchunks = (bn + 31) >> 5;
      const int oc0 = __ldg(g.out_col);
      const int ac0 = g.addend ? (g.add_col ? __ldg(g.add_col) : oc0) : 0;
      // The four output rows this thread stores, their table entries and the column bases are fetched while the main
      // loop still runs (they sat on the critical path of every chunk before).  out_vec contract: the column tables are
      // contiguous, col[n] = col[0] + n.
      int r_out[TC_BM / 32], r_add[TC_BM / 32], r_aux[TC_BM / 32];
      bool r_ok[TC_BM / 32];
#pragma unroll
      for (int it = 0; it < TC_BM / 32; ++it) {
        const int m = m0 + it * 32 + ew * 4 + rsub;
        r_ok[it] = m < m_lim;
        r_out[it] = r_add[it] = r_aux[it] = 0;
        if (r_ok[it]) {
          const EpiRow er = epi_row(g, m);
          r_out[it] = er.out; r_add[it] = er.add;
          r_aux[it] = g.aux_out ? (g.aux_row ? __ldg(g.aux_row + m) : er.out) : 0;
        }
      }
      // bias of this tile's columns: fetched now, read back from shared memory after the chunk barriers (a global load
      // per chunk sat on the critical path of the store phase: 1650 of a chunk's 2270 clocks, profiles/timeline_*_r02m)
      if (g.bias && !atomic)
        for (int i = tid - 64; i < bn; i += TM_THREADS - 64) sh->bias[i] = n0 + i < g.N ? __ldg(g.bias + n0 + i) : 0.f;
      split_loop();
      if (tid == 64) TL_STAMP(5);                                // last residual tile written
      mbar_wait(smem_u32(&sh->accum_full), 0u);
      tc_fence_after();
      if (tid == 64) TL_STAMP(6);                                // accumulator complete
      // Software pipeline over 32-column chunks: the TMEM loads of chunk c + 1 (all partial accumulators, one wait) are
      // in flight while chunk c is stored, and the gate / residual operands of chunk c while its columns are staged.
      constexpr int NA = X3 ? 5 : 1;
      uint32_t acc[NA][16];
      auto drain_issue = [&](int c) {
        if (c * 32 + half * 16 < bn) {
          const uint32_t ta = tmem_d + ((uint32_t)(quad * 32) << 16) + (uint32_t)(c * 32 + half * 16);
#pragma unroll
          for (int a = 0; a < NA; ++a)
            if (a < n_acc) tmem_ld16_issue(ta + (uint32_t)a * acc_stride, acc[a]);
        }
      };
      drain_issue(0);
      for (int c = 0; c < nchunks; ++c) {
        const uint32_t stg = stg0 + (uint32_t)(c & 1) * (TC_BM * TM_EPI_PITCH * 4);
        const int n = n0 + c * 32 + cq * 4;
        const bool nvalid = n < g.N && c * 32 + cq * 4 < bn;
        const bool gated = g.gate && n >= g.gate_col0;
        float4 gt[TC_BM / 32], ad[TC_BM / 32];
#pragma unroll
        for (int it = 0; it < TC_BM / 32; ++it) {
          gt[it] = make_float4(1.f, 1.f, 1.f, 1.f);
          ad[it] = f4zero();
          if (nvalid && r_ok[it] && !atomic) {
            if (gated) gt[it] = ldg128(g.gate + (r_out[it] + oc0 + n));
            if (g.addend) ad[it] = ldg128(g.addend + (r_add[it] + ac0 + n));
          }
        }
        if (c * 32 + half * 16 < bn) {
          tmem_ld_wait();
          float v[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(acc[0][j]);
#pragma unroll
          for (int a = 1; a < NA; ++a)
            if (a < n_acc) {
#pragma unroll
              for (int j = 0; j < 16; ++j) v[j] += __uint_as_float(acc[a][j]);
            }
          if (tid == 64 && c == 1) TL_STAMP(8);                  // chunk 1: accumulator columns in registers
          const uint32_t dst = stg + (uint32_t)(trow * TM_EPI_PITCH + half * 16) * 4;
#pragma unroll
          for (int j = 0; j < 16; j += 4) sts128(dst + j * 4, v[j], v[j + 1], v[j + 2], v[j + 3]);
        }
        if (tid == 64 && c == 1) TL_STAMP(9);                    // staged
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (tid == 64 && c == 1) TL_STAMP(10);                   // all warps staged
        if (c + 1 < nchunks) drain_issue(c + 1);
        if (nvalid) {
          float4 bias4 = f4zero();
          if (g.bias && !atomic) bias4 = *reinterpret_cast<const float4*>(&sh->bias[c * 32 + cq * 4]);
#pragma unroll
          for (int it = 0; it < TC_BM / 32; ++it) {
            if (!r_ok[it]) continue;
            const int row = it * 32 + ew * 4 + rsub;
            float4 v;
            asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];"
                         : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                         : "r"(stg + (uint32_t)(row * TM_EPI_PITCH + cq * 4) * 4));
            float* o = g.out + (r_out[it] + oc0 + n);
            if (atomic) {
              asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(o), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
              continue;
            }
            *reinterpret_cast<float4*>(o) = epi_final4(g, v, n, bias4, gt[it], ad[it], gated, r_out[it] + oc0, r_aux[it]);
          }
        }
        if (tid == 64 && c == 0) TL_STAMP(11);                   // chunk 0 stored = chunk 1 begins
        if (tid == 64 && c == 1) TL_STAMP(12);                   // chunk 1 stored
      }
      if (atomic && g.finish_counter) splitk_finish(g, &sh->last_flag, tid - 64, m0, m_lim, n0, bn);
    } else if (g.out_vec == 2) {
      split_loop();
      mbar_wait(smem_u32(&sh->accum_full), 0u);
      tc_fence_after();
      epi_rows_contiguous(g, smem_base, tmem_d, n_acc, acc_stride, bn, m0, n0, quad, half, ew, lane, atomic);
    } else {
      const int m = m0 + quad * 32 + lane;
      const bool mvalid = m < m_lim;
      EpiRow er = {0, 0, false};
      if (mvalid) er = epi_row(g, m);
      split_loop();
      mbar_wait(smem_u32(&sh->accum_full), 0u);
      tc_fence_after();
      const int nchunks = bn >> 4;
      for (int c = half; c < nchunks; c += 2) {
        float v[16];
        const uint32_t ta = tmem_d + ((uint32_t)(quad * 32) << 16) + (uint32_t)(c * 16);
        tmem_ld16_sum(ta, n_acc, acc_stride, v);
        if (mvalid) {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int n = n0 + c * 16 + j;
            if (n < g.N) epi_store(g, er, n, v[j], atomic);
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (tid == 0) TL_STAMP(7);                                     // epilogue done
  if (warp == 1) {
    __syncwarp();
    tmem_dealloc(tmem_d, (uint32_t)tmem_cols);
  }
}

// ---------------------------------------------------------------------------- host
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
typedef CUresult (*EncodeIm2colFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const int*, const int*, cuuint32_t, cuuint32_t, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int driver_fn(const char* name, void** fn) {
  cudaDriverEntryPointQueryResult q;
  cudaError_t e = cudaGetDriverEntryPoint(name, fn, cudaEnableDefault, &q);
  if (e != cudaSuccess) return cuda_check(e, name);
  if (q != cudaDriverEntryPointSuccess || *fn == nullptr) return fail(OFFK_E_NOTSM100, "%s: driver entry point unavailable", name);
  return 0;
}

static int encode_2d(CUtensorMap* tm, const float* base, long long inner, long long rows, long long ld, int box_rows,
                     bool mn_major = false) {
  static EncodeTiledFn fn = nullptr;
  if (!fn)
    if (int e = driver_fn("cuTensorMapEncodeTiled", (void**)&fn)) return e;
  const cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
  const cuuint32_t box[2] = {(cuuint32_t)TC_BK, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(OFFK_E_BADARG, "cuTensorMapEncodeTiled failed (%d): inner=%lld rows=%lld ld=%lld box=%d", (int)r, inner, rows, ld, box_rows);
  return 0;
}

// Weights with their tf32 residuals split ahead of time: [N, ldb] matrix at base (plane 0) and its residual matrix `delta`
// elements further (plane 1), as one 3-D map {K, N, 2}; box {32 k, bn rows, 1 plane}
static int encode_b_planes(CUtensorMap* tm, const float* base, long long K, long long N, long long ld, int box_rows, long long delta) {
  static EncodeTiledFn fn = nullptr;
  if (!fn)
    if (int e = driver_fn("cuTensorMapEncodeTiled", (void**)&fn)) return e;
  const cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)N, 2};
  const cuuint64_t strides[2] = {(cuuint64_t)ld * 4, (cuuint64_t)delta * 4};
  const cuuint32_t box[3] = {(cuuint32_t)TC_BK, (cuuint32_t)box_rows, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(OFFK_E_BADARG, "cuTensorMapEncodeTiled(B planes) failed (%d): K=%lld N=%lld ld=%lld delta=%lld", (int)r, K, N, ld, delta);
  return 0;
}

// NCHW [n_img, cin, hw] as {hw, cin, n_img}; box {32 pixels, 32 channels, 1 frame}; 32-byte-atom 128B swizzle = the
// MN-major SWIZZLE_128B_BASE32B operand layout of kind::tf32 (cute Swizzle<2,5,2>)
static int encode_nchw(CUtensorMap* tm, const float* base, long long hw, long long cin, long long n_img, bool transposed) {
  static EncodeTiledFn fn = nullptr;
  if (!fn)
    if (int e = driver_fn("cuTensorMapEncodeTiled", (void**)&fn)) return e;
  const cuuint64_t dims[3] = {(cuuint64_t)hw, (cuuint64_t)cin, (cuuint64_t)n_img};
  const cuuint64_t strides[2] = {(cuuint64_t)hw * 4, (cuuint64_t)hw * cin * 4};
  // forward (m = pixel): {32 pixels, 32 channels} MN-major atoms; transposed (m = channel, k = pixel): one K-major
  // {32 pixels, 128 channels} tile
  const cuuint32_t box[3] = {32, (cuuint32_t)(transposed ? TC_BM : TC_BK), 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, transposed ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(OFFK_E_BADARG, "cuTensorMapEncodeTiled(nchw) failed (%d): hw=%lld cin=%lld n=%lld", (int)r, hw, cin, n_img);
  return 0;
}

// Output rows [rows, ld] (or [n_img, rows, ld] when n_img > 0: per-frame tiles clip at the frame end), columns [0, ncols) of
// the slice at `base`; box {32 columns, 128 rows}, SWIZZLE_128B: the staging layout of the TMA-store epilogue
static int encode_out(CUtensorMap* tm, const float* base, long long ncols, long long rows, long long n_img, long long ld) {
  static EncodeTiledFn fn = nullptr;
  if (!fn)
    if (int e = driver_fn("cuTensorMapEncodeTiled", (void**)&fn)) return e;
  const cuuint64_t dims[3] = {(cuuint64_t)ncols, (cuuint64_t)rows, (cuuint64_t)(n_img > 0 ? n_img : 1)};
  const cuuint64_t strides[2] = {(cuuint64_t)ld * 4, (cuuint64_t)rows * ld * 4};
  const cuuint32_t box[3] = {32, (cuuint32_t)TC_BM, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, n_img > 0 ? 3 : 2, const_cast<float*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(OFFK_E_BADARG, "cuTensorMapEncodeTiled(out) failed (%d): ncols=%lld rows=%lld ld=%lld", (int)r, ncols, rows, ld);
  return 0;
}

static int encode_im2col(CUtensorMap* tm, const offk_tgemm_t* t, bool transposed, int bk) {
  static EncodeIm2colFn fn = nullptr;
  if (!fn)
    if (int e = driver_fn("cuTensorMapEncodeIm2col", (void**)&fn)) return e;
  const cuuint64_t dims[4] = {(cuuint64_t)t->ctot, (cuuint64_t)t->win, (cuuint64_t)t->hin, (cuuint64_t)t->n_img};
  const cuuint64_t strides[3] = {(cuuint64_t)t->ctot * 4, (cuuint64_t)t->win * t->ctot * 4,
                                 (cuuint64_t)t->hin * t->win * t->ctot * 4};
  // base pixels (top-left corner of the filter window) range over [-pad, dim + pad - (k - 1)) in steps of `stride`
  int lower[2] = {-t->pad, -t->pad};
  int upper[2] = {t->pad - (t->kw - 1), t->pad - (t->kh - 1)};
  if (t->geom_flags & OFFK_TGEMM_FREE_GEOM) {
    // caller-given output grid and top / left padding (data gradient of a strided conv as a stride-1 correlation over
    // dY): base pixels run from -pad to -pad + (n_out - 1) * stride, whatever that implies for the bottom / right edge
    lower[0] = -t->pad_w; lower[1] = -t->pad;
    upper[0] = (t->wout - 1) * t->stride - t->pad_w - (t->win - 1);
    upper[1] = (t->hout - 1) * t->stride - t->pad - (t->hin - 1);
  }
  const cuuint32_t estr[4] = {1, (cuuint32_t)t->stride, (cuuint32_t)t->stride, 1};
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(t->g.a_src), dims, strides, lower, upper,
                  (cuuint32_t)TC_BK, (cuuint32_t)(transposed ? bk : TC_BM), estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  transposed ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(OFFK_E_BADARG, "cuTensorMapEncodeIm2col failed (%d): [n=%d h=%d w=%d c=%d] k=%dx%d s=%d p=%d", (int)r, t->n_img,
                t->hin, t->win, t->ctot, t->kh, t->kw, t->stride, t->pad);
  return 0;
}

template <int A_KIND, int B_KIND, bool X3>
static int launch_tm_t(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const offk_gemm_t& g, const TmGeom& geo, int bn,
                       int stages, int kb_per, int tmem_cols, int n_main, int bk, int b_presplit, int a_tmem, int c_mode, dim3 grid,
                       size_t smem, cudaStream_t st) {
  auto kern = tma_gemm_kernel<A_KIND, B_KIND, X3>;
  static bool attr_set = false;  // per instantiation
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return cuda_check(e, "cudaFuncSetAttribute(tma_gemm)");
    attr_set = true;
  }
  cudaError_t e = launch_pdl(kern, grid, dim3(TM_THREADS), smem, st, ta, tb, tc, g, geo, bn, stages, kb_per, tmem_cols, n_main,
                             bk, b_presplit, a_tmem, c_mode);
  if (e != cudaSuccess) return cuda_check(e, "tma_gemm launch");
  return OFFK_LAUNCH_CHECK("tma_gemm");
}

}  // namespace offk

using namespace offk;

namespace offk {
__global__ void __launch_bounds__(256) tf32_residual_kernel(const float* __restrict__ src, float* __restrict__ dst, long long n4) {
  pdl_sync();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  const float4 v = __ldg(reinterpret_cast<const float4*>(src) + i);
  reinterpret_cast<float4*>(dst)[i] = make_float4(tf32_lo(v.x), tf32_lo(v.y), tf32_lo(v.z), tf32_lo(v.w));
}
}  // namespace offk

extern "C" int offk_tf32_residual(const float* src, float* dst, long long n, void* stream) {
  OFFK_REQUIRE(src && dst && n > 0 && n % 4 == 0, "tf32_residual: n must be a positive multiple of 4");
  OFFK_REQUIRE(((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15u) == 0, "tf32_residual: alignment");
  const long long n4 = n / 4;
  cudaError_t e = launch_pdl(tf32_residual_kernel, dim3((unsigned)((n4 + 255) / 256)), dim3(256), 0, as_stream(stream), src, dst, n4);
  if (e != cudaSuccess) return cuda_check(e, "tf32_residual launch");
  return OFFK_LAUNCH_CHECK("tf32_residual");
}

extern "C" int offk_tma_gemm_prepare(offk_tgemm_t* t) {
  OFFK_REQUIRE(t != nullptr, "tma_gemm: null descriptor");
  const offk_gemm_t& g = t->g;
  OFFK_REQUIRE(g.M > 0 && g.N > 0 && g.K > 0, "tma_gemm: empty problem");
  OFFK_REQUIRE(g.a_src && g.b_src, "tma_gemm: operand pointers");
  OFFK_REQUIRE((reinterpret_cast<uintptr_t>(g.a_src) & 15u) == 0 && (reinterpret_cast<uintptr_t>(g.b_src) & 15u) == 0,
               "tma_gemm: operands must be 16-byte aligned");
  const bool wgrad = (t->a_kind == OFFK_TMA_A_NCHW_T || t->a_kind == OFFK_TMA_A_IM2COL_T);
  OFFK_REQUIRE(wgrad == (t->b_kind == OFFK_TMA_B_DENSE_T), "tma_gemm: transposed A kinds pair with OFFK_TMA_B_DENSE_T and only with it");
  int bn = g.tile_n > 0 ? g.tile_n : (g.N <= 256 ? (g.N + 15) / 16 * 16 : 256);
  OFFK_REQUIRE(bn % 16 == 0 && bn >= 16 && bn <= 256, "tma_gemm: bad N tile %d", bn);
  const int bk = t->bk > 0 ? t->bk : TC_BK;
  OFFK_REQUIRE(bk == 32 || ((bk == 64 || bk == 128) && t->a_kind == OFFK_TMA_A_IM2COL_T),
               "tma_gemm: bk is 32, or 64 / 128 for OFFK_TMA_A_IM2COL_T (both operands MN-major)");
  const long long hw = (long long)t->hin * t->win;
  CUtensorMap ta, tb;
  if (t->a_kind == OFFK_TMA_A_DENSE) {
    OFFK_REQUIRE(t->lda >= g.K && t->lda % 4 == 0, "tma_gemm: dense A needs lda >= K, lda %% 4 == 0");
    if (int e = encode_2d(&ta, g.a_src, g.K, g.M, t->lda, TC_BM)) return e;
  } else if (t->a_kind == OFFK_TMA_A_IM2COL || t->a_kind == OFFK_TMA_A_IM2COL_T) {
    OFFK_REQUIRE(t->cin % TC_BK == 0 && t->ctot % 4 == 0 && t->a_coff % 4 == 0 && t->a_coff + t->cin <= t->ctot,
                 "tma_gemm: im2col needs cin %% 32 == 0 and a 16-byte aligned channel slice");
    OFFK_REQUIRE(t->kh >= 1 && t->kw >= 1 && t->stride >= 1 && t->stride <= 8 && t->pad >= 0, "tma_gemm: conv geometry");
    if (t->geom_flags & OFFK_TGEMM_FREE_GEOM) {
      OFFK_REQUIRE(t->a_kind == OFFK_TMA_A_IM2COL && t->pad_w >= 0 && t->hout >= 1 && t->wout >= 1, "tma_gemm: free geometry is for im2col A");
    } else {
      OFFK_REQUIRE(t->hout == (t->hin + 2 * t->pad - t->kh) / t->stride + 1 && t->wout == (t->win + 2 * t->pad - t->kw) / t->stride + 1,
                   "tma_gemm: output geometry");
    }
    const long long pixels = (long long)t->n_img * t->hout * t->wout, kw_rows = (long long)t->cin * t->kh * t->kw;
    if (t->a_kind == OFFK_TMA_A_IM2COL) {
      OFFK_REQUIRE(g.K == kw_rows && g.M == pixels, "tma_gemm: im2col needs K == kh*kw*cin, M == output pixels");
    } else {
      OFFK_REQUIRE(g.K == pixels && (g.M == kw_rows || (g.M == kw_rows + 1 && g.a_ones_row == kw_rows)),
                   "tma_gemm: im2col_t needs K == output pixels, M == kh*kw*cin (+ the ones row)");
    }
    if (int e = encode_im2col(&ta, t, t->a_kind == OFFK_TMA_A_IM2COL_T, bk)) return e;
  } else if (t->a_kind == OFFK_TMA_A_NCHW) {
    OFFK_REQUIRE(hw % 4 == 0 && t->cin % TC_BK == 0 && g.K == t->cin && g.M == (long long)t->n_img * hw && t->ctot == t->cin,
                 "tma_gemm: nchw A needs hw %% 4 == 0, cin %% 32 == 0, K == cin, M == n_img*hw");
    if (int e = encode_nchw(&ta, g.a_src, hw, t->cin, t->n_img, false)) return e;
  } else if (t->a_kind == OFFK_TMA_A_NCHW_T) {
    OFFK_REQUIRE(hw % 4 == 0 && t->ctot == t->cin && g.K == (long long)t->n_img * hw &&
                     (g.M == t->cin || (g.M == t->cin + 1 && g.a_ones_row == t->cin)),
                 "tma_gemm: nchw_t A needs hw %% 4 == 0, K == n_img*hw, M == cin (+ the ones row)");
    if (int e = encode_nchw(&ta, g.a_src, hw, t->cin, t->n_img, true)) return e;
  } else {
    return fail(OFFK_E_BADARG, "tma_gemm: unknown a_kind %d", t->a_kind);
  }
  if (t->b_kind == OFFK_TMA_B_DENSE) {
    OFFK_REQUIRE(t->ldb >= g.K && t->ldb % 4 == 0, "tma_gemm: B must be a dense [N, ldb] matrix, ldb %% 4 == 0");
    if (t->precision == OFFK_PREC_TF32X3 && t->b_lo_delta != 0) {
      OFFK_REQUIRE(t->b_lo_delta > 0 && t->b_lo_delta % 4 == 0, "tma_gemm: b_lo_delta must be a positive multiple of 4 elements");
      if (int e = encode_b_planes(&tb, g.b_src, g.K, g.N, t->ldb, bn, t->b_lo_delta)) return e;
    } else if (int e = encode_2d(&tb, g.b_src, g.K, g.N, t->ldb, bn)) return e;
  } else if (t->b_kind == OFFK_TMA_B_DENSE_T) {
    OFFK_REQUIRE(t->ldb >= g.N && t->ldb % 4 == 0, "tma_gemm: transposed B must be a row-major [K, ldb] matrix, ldb %% 4 == 0");
    if (int e = encode_2d(&tb, g.b_src, g.N, g.K, t->ldb, bk, true)) return e;     // {32 n, bk k} stacks of atoms
  } else {
    return fail(OFFK_E_BADARG, "tma_gemm: unknown b_kind %d", t->b_kind);
  }
  memcpy(t->tmap_a, &ta, sizeof(ta));
  memcpy(t->tmap_b, &tb, sizeof(tb));
  t->c_mode = 0;
  if (t->out_ld > 0 && g.out_vec == 1 && !wgrad) {
    OFFK_REQUIRE(t->out_ld % 4 == 0 && t->out_c0 % 4 == 0 && t->out_c0 >= 0 && t->out_c0 + g.N <= t->out_ld,
                 "tma_gemm: out_ld / out_c0 must describe a 16-byte aligned column slice of the output rows");
    CUtensorMap tc;
    if (int e = encode_out(&tc, g.out + t->out_c0, g.N, t->a_kind == OFFK_TMA_A_NCHW ? hw : (long long)g.M,
                           t->a_kind == OFFK_TMA_A_NCHW ? t->n_img : 0, t->out_ld))
      return e;
    memcpy(t->tmap_c, &tc, sizeof(tc));
    t->c_mode = t->a_kind == OFFK_TMA_A_NCHW ? 2 : 1;
  }
  t->prepared = bn;
  return 0;
}

extern "C" int offk_tma_gemm(const offk_tgemm_t* t, void* stream) {
  OFFK_REQUIRE(t != nullptr && t->prepared > 0, "tma_gemm: descriptor not prepared (offk_tma_gemm_prepare)");
  const offk_gemm_t& g = t->g;
  OFFK_REQUIRE(g.out && g.out_row && g.out_col, "tma_gemm: output tables");
  if (g.out_vec == 1) OFFK_REQUIRE((g.N & 3) == 0 && (reinterpret_cast<uintptr_t>(g.out) & 15u) == 0, "tma_gemm: out_vec alignment");
  if (g.out_vec == 2)
    OFFK_REQUIRE((reinterpret_cast<uintptr_t>(g.out) & 15u) == 0 && !g.bias && !g.gate && !g.addend && !g.relu_pre_cols && !g.relu_post,
                 "tma_gemm: out_vec = 2 needs a 16-byte aligned `out` and a plain epilogue");
  OFFK_REQUIRE(g.out_vec == 1 || (!g.finish_counter && !g.aux_out), "tma_gemm: finish_counter / aux_out need out_vec = 1");
  OFFK_REQUIRE(!g.finish_counter || (g.split_k > 1 && !g.atomic_out), "tma_gemm: finish_counter is for split_k > 1 without atomic_out");
  OFFK_REQUIRE(!g.aux_out || g.finish_counter || (g.split_k <= 1 && !g.atomic_out), "tma_gemm: aux_out needs a final value (no raw accumulation)");
  if (g.aux_out) OFFK_REQUIRE((reinterpret_cast<uintptr_t>(g.aux_out) & 15u) == 0, "tma_gemm: aux_out alignment");
  const int bn = t->prepared;
  TmGeom geo;
  geo.a_kind = t->a_kind; geo.a_coff = t->a_coff; geo.cblocks = t->cin > 0 ? t->cin / TC_BK : 1; geo.kw = t->kw > 0 ? t->kw : 1;
  geo.hout = t->hout; geo.wout = t->wout; geo.stride = t->stride; geo.pad = t->pad;
  geo.pad_w = (t->geom_flags & OFFK_TGEMM_FREE_GEOM) ? t->pad_w : t->pad;
  geo.hw = t->hin * t->win; geo.tiles_per_img = (geo.hw + TC_BM - 1) / TC_BM;
  geo.kb_per_img = (geo.hw + TC_BK - 1) / TC_BK;
  geo.kw_rows = t->cin * t->kh * t->kw;
  const bool wgrad = t->b_kind == OFFK_TMA_B_DENSE_T;
  OFFK_REQUIRE(!(wgrad && g.out_vec == 1), "tma_gemm: weight-gradient kinds write rows, not columns (out_vec = 0 or 2)");
  OFFK_REQUIRE(g.out_vec != 2 || t->a_kind != OFFK_TMA_A_NCHW, "tma_gemm: out_vec = 2 with per-frame M tiles");
  const int bk = t->bk > 0 ? t->bk : TC_BK;
  const int num_kb = t->a_kind == OFFK_TMA_A_NCHW_T ? t->n_img * geo.kb_per_img : (g.K + bk - 1) / bk;
  const int split = g.split_k > 1 ? g.split_k : 1;
  const int kb_per = (num_kb + split - 1) / split;
  const uint32_t a_bytes = t->a_kind == OFFK_TMA_A_IM2COL_T ? (uint32_t)bk * 512u : (uint32_t)TC_A_BYTES;
  const uint32_t b_bytes = wgrad ? (uint32_t)((bn + 31) / 32) * (uint32_t)bk * 128u : (uint32_t)bn * 128u;
  OFFK_REQUIRE(t->precision == 0 || t->precision == OFFK_PREC_TF32 || t->precision == OFFK_PREC_TF32X3,
               "tma_gemm: precision must be OFFK_PREC_TF32 (or 0) or OFFK_PREC_TF32X3");
  const bool x3 = t->precision == OFFK_PREC_TF32X3;
  const int presplit = (x3 && t->b_kind == OFFK_TMA_B_DENSE && t->b_lo_delta != 0) ? 1 : 0;
  // 3xTF32 with the A operand in tensor memory (kernel comment): possible when the accumulators leave room for at least
  // two (A_hi, A_lo) column pairs; the wide tiles (N tile > 192) keep both operands in shared memory.  One CTA per SM.
  const int acc_stride = (bn + 31) / 32 * 32;
  const int a_cols = t->a_kind == OFFK_TMA_A_IM2COL_T ? bk : TC_BK;
  const int mmas = kb_per * (bk / 8);                      // K = 8 steps per output tile
  int atm = 0, atm_main = 0, atm_slots = 0;
  if (x3) {
    // chains of at most 64 MMAs per main accumulator where tensor memory has the room (measured: the chain policy does
    // not move the step time -- profiles/env_r02x.log -- but single 800-MMA chains took the fc14 error from 3.7e-6 to
    // 6.7e-6)
    constexpr int chain = 64;
    const int want = x3_main_accumulators(4, (mmas * 64 + chain - 1) / chain);
    for (int nm = want; nm >= 1 && !atm; --nm) {
      const int slots = (512 - (1 + nm) * acc_stride) / (2 * a_cols);
      if (slots >= 2) { atm = 1; atm_main = nm; atm_slots = slots; }
    }
  }
  const uint32_t stage_bytes = atm ? a_bytes + 2u * b_bytes : (a_bytes + b_bytes) * (x3 ? 2u : 1u);   // x3: residual tiles
  OFFK_REQUIRE(2 * stage_bytes <= 216u * 1024u, "tma_gemm: a pipeline stage of %u bytes leaves no room for two (N tile %d, bk %d)", stage_bytes, bn, bk);
  // two CTAs per SM (one CTA's epilogue overlaps the other's main loop) when that still leaves a pipeline; the 3xTF32
  // stages and the deep K-blocks of the wide tiles need the whole SM
  int budget = 108 * 1024;
  if (atm || 2 * stage_bytes > (uint32_t)budget || (x3 && 3 * stage_bytes > (uint32_t)budget)) budget = 216 * 1024;
  int stages = budget / (int)stage_bytes;
  if (stages < 2) stages = 2;
  if (stages > TC_MAX_STAGES) stages = TC_MAX_STAGES;
  if (stages > kb_per) stages = kb_per < 2 ? 2 : kb_per;
  size_t pipe_bytes = (size_t)stages * stage_bytes;
  int n_main = 1, tmem_need = bn;
  if (atm) {
    n_main = atm_main;
    if (atm_slots > stages) atm_slots = stages;
    tmem_need = (1 + n_main) * acc_stride + atm_slots * 2 * a_cols;
  } else if (x3) {
    // TMEM columns: 256 per CTA while two CTAs share the SM, all 512 otherwise; (n_main + 1) accumulators of bn columns
    // (32-column granules), at most 4 mains (see tmem_ld16_sum)
    const int cap = budget > 108 * 1024 ? 512 : 256, stride = acc_stride;
    n_main = cap / stride - 1;
    if (n_main > 4) n_main = 4;
    n_main = x3_main_accumulators(n_main, mmas);
    OFFK_REQUIRE(n_main >= 1, "tma_gemm: no room in tensor memory for the 3xTF32 accumulators (N tile %d)", bn);
    tmem_need = (n_main + 1) * stride;
  }
  int tmem_cols = 32;
  while (tmem_cols < tmem_need) tmem_cols <<= 1;
  dim3 grid((g.M + TC_BM - 1) / TC_BM, (g.N + bn - 1) / bn, (num_kb + kb_per - 1) / kb_per);
  if (t->a_kind == OFFK_TMA_A_NCHW) grid.x = (unsigned)(t->n_img * geo.tiles_per_img);
  OFFK_REQUIRE(grid.y <= 65535 && grid.z <= 65535, "tma_gemm: grid too large");
  alignas(64) CUtensorMap ta, tb, tc;
  memcpy(&ta, t->tmap_a, sizeof(ta));
  memcpy(&tb, t->tmap_b, sizeof(tb));
  memcpy(&tc, t->tmap_c, sizeof(tc));
  // TMA stores (offk.h: out_ld) for plain epilogues only: bias / ReLU, or split-K partial sums.  Measured -3.4 % (fp32) /
  // -2.5 % (tf32) of the step against st.global everywhere; a second pass over the slab for the ReLU' gate and residual
  // addend bought nothing on top (profiles/env_r03f-i.log): its barrier and shared-memory pass cost what the faster
  // stores save.
  const int c_mode = (t->c_mode && g.out_vec == 1 && !g.finish_counter && !g.aux_out && bn % 32 == 0 && !g.gate && !g.addend)
                         ? t->c_mode : 0;
  // same formula as the kernel: the shared structure follows max(pipeline stages, epilogue staging)
  const size_t epi_bytes = c_mode ? 3 * TC_BM * 128 : 2 * TC_BM * TM_EPI_PITCH * 4;
  if (pipe_bytes < epi_bytes) pipe_bytes = epi_bytes;
  size_t smem = pipe_bytes + sizeof(TmShared) + 1024;
  if (atm && smem < 120 * 1024) smem = 120 * 1024;          // the whole tensor memory is ours: keep a second CTA off the SM
  cudaStream_t st = as_stream(stream);
#define OFFK_TM_CASE(AK, BK)                                                                                          \
  if (t->a_kind == AK && t->b_kind == BK)                                                                             \
    return x3 ? launch_tm_t<AK, BK, true>(ta, tb, tc, g, geo, bn, stages, kb_per, tmem_cols, n_main, bk, presplit, atm ? atm_slots : 0, c_mode, grid, smem, st)  \
              : launch_tm_t<AK, BK, false>(ta, tb, tc, g, geo, bn, stages, kb_per, tmem_cols, n_main, bk, 0, 0, c_mode, grid, smem, st);
  OFFK_TM_CASE(OFFK_TMA_A_DENSE, OFFK_TMA_B_DENSE)
  OFFK_TM_CASE(OFFK_TMA_A_IM2COL, OFFK_TMA_B_DENSE)
  OFFK_TM_CASE(OFFK_TMA_A_NCHW, OFFK_TMA_B_DENSE)
  OFFK_TM_CASE(OFFK_TMA_A_NCHW_T, OFFK_TMA_B_DENSE_T)
  OFFK_TM_CASE(OFFK_TMA_A_IM2COL_T, OFFK_TMA_B_DENSE_T)
#undef OFFK_TM_CASE
  return fail(OFFK_E_BADARG, "tma_gemm: unsupported operand kinds %d/%d", t->a_kind, t->b_kind);
}

#ifdef OFFK_TIMELINE
// diagnostics build only: fetch / clear the per-CTA phase stamps (not part of include/offk.h)
extern "C" int offk_timeline_read(long long* host, int n_ctas) {
  if (n_ctas > offk::TL_MAX_CTAS) n_ctas = offk::TL_MAX_CTAS;
  return (int)cudaMemcpyFromSymbol(host, offk::tl_buf, sizeof(long long) * n_ctas * offk::TL_SLOTS);
}
extern "C" int offk_timeline_clear() {
  void* p = nullptr;
  cudaGetSymbolAddress(&p, offk::tl_buf);
  return (int)cudaMemset(p, 0, sizeof(offk::tl_buf));
}
#endif
