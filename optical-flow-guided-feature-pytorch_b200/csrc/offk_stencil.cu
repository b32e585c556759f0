// Fused OFF stencil kernels (forward and backward) on channels-last tensors; HBM-bound by construction.
//
// One launch serves a BATCH of OFF units (the units feeding one stage-fusion buffer, or all nine in the backward
// pass), so the 14x14 and 7x7 levels -- a few MB each -- do not pay one launch latency apiece.  A block is either
//   a temporal block : (clip, 64 pixels).  One warp = the 128 reduced channels of a pixel (lane = channel quad), so
//                      there is no index arithmetic beyond pointer increments.  A warp walks 4 pixel pairs; for each
//                      pair every frame is read exactly once (128-bit loads, 512 contiguous bytes per warp), all
//                      frames of the pair in flight together (L = 3) or two frames ahead (general L), and every
//                      difference G(t+1) - G(t) is written once.
//   a spatial block  : (pair, band of rows).  The D band plus a one-pixel halo is staged in shared memory with
//                      16-byte cp.async (zero-fill gives the conv's zero padding); each thread then produces two
//                      horizontally adjacent (pixel, 4 channels) outputs from twelve LDS.128 neighbours with the
//                      per-channel taps held in registers; bias, dropout and the stores at the unit's channel offset
//                      of the stage buffer follow.  K = 2 emits two maps per channel (Sobel x and y).
// Spatial blocks (instruction-heavy, few bytes) are spread evenly between the temporal blocks (streaming) of their
// level.  No torch.cat, no sub, no conv2d, no separate dropout launch.
//
// Backward mirrors it: dG = (dT(t-1) - dT(t)) * [G > 0]; the spatial blocks stage the DROPPED spatial gradient dS
// (band + halo) once and use the same nine neighbours twice: dD = transposed stencil of dS, and
// dw[a,b] += D(y,x) * dS(y-a+1, x-b+1) (the tap gradient re-indexed so that it needs D only at the centre pixel).
// Tap / bias gradients are accumulated in registers over a few consecutive items, reduced with warp shuffles and
// shared-memory atomics, then one global atomicAdd per tap and block.
#include "offk_common.cuh"

namespace offk {

constexpr int ST_FWD_MINB = 3;   // resident blocks per SM the kernels are compiled for (register cap 80; 4 spills, DESIGN 3.1)
constexpr int ST_THREADS = 256;
constexpr int ST_WARPS = ST_THREADS / 32;
constexpr int ST_MAX_LEVELS = 12;
constexpr int ST_MAX_CS = 64;                 // spatial channels per level (32 on the path)
constexpr int ST_TIT = 4;                     // pixel pairs per warp: a temporal block covers ST_WARPS*2*ST_TIT = 64 pixels
constexpr int ST_TPIX = ST_WARPS * 2 * ST_TIT;
constexpr int ST_WQ = 16;                     // channel quads per tap row in shared memory (= ST_MAX_CS / 4)
constexpr int ST_ITEMS = 8;                   // max (frame, band) items per backward spatial block
constexpr int ST_TILE_BUDGET = 24 * 1024;     // target size of a halo tile (bytes)
constexpr int ST_SMEM_MAX = 64 * 1024;

struct StLevel {
  offk_stencil_t s;
  const float* g;
  const float* d;
  const float* w;
  const float* bias;
  float* out;          // forward: stage buffer
  const float* dout;   // backward: gradient of the stage buffer
  float* dg;
  float* dd;
  float* dw;
  float* dbias;
  long long dg_fs, dd_fs;
  int blk0;            // first block of this level
  int n_sblocks;       // spatial blocks
  int n_sitems;        // spatial items = (pair | frame) x band
  int n_tblocks;       // temporal blocks
  int lstride;         // log2 spacing of the spatial blocks inside the level's block range
  int bands, band_rows;
  int t_chunks;        // temporal blocks per clip
  int ipb;             // backward: (frame, band) items per spatial block
  int lq, ltcp;        // log2: channel quads per pixel, tile column pitch
  int lpw;             // forward: log2 pixel-PAIR slots per row and pass
  int lxw;             // backward: log2 pixel slots per row and pass
};
struct StBatch {
  int n;
  StLevel lv[ST_MAX_LEVELS];
};

__device__ __forceinline__ float4 f4sub(float4 a, float4 b) { return make_float4(a.x - b.x, a.y - b.y, a.z - b.z, a.w - b.w); }
__device__ __forceinline__ float4 f4zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ float4 f4mul(float4 a, float4 b) { return make_float4(a.x * b.x, a.y * b.y, a.z * b.z, a.w * b.w); }
__device__ __forceinline__ void f4fma(float4& acc, float4 w, float4 v) {
  acc.x = fmaf(w.x, v.x, acc.x);
  acc.y = fmaf(w.y, v.y, acc.y);
  acc.z = fmaf(w.z, v.z, acc.z);
  acc.w = fmaf(w.w, v.w, acc.w);
}
__device__ __forceinline__ float4 relu_gate4(float4 g, float4 r) {
  return make_float4(g.x > 0.f ? r.x : 0.f, g.y > 0.f ? r.y : 0.f, g.z > 0.f ? r.z : 0.f, g.w > 0.f ? r.w : 0.f);
}
__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ uint32_t st_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void st_cp_async16(uint32_t dst, const float* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void st_cp_async_wait_all() {
  asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
}

__device__ __forceinline__ int spatial_frame(const offk_stencil_t& s, int p) {
  if (s.index_mode == OFFK_INDEX_REFERENCE_FLAT) return p;
  const int b = p / (s.L - 1), t = p - b * (s.L - 1);
  return b * s.L + t;
}
// pair fed by frame f through the spatial branch, or -1
__device__ __forceinline__ int spatial_pair_of_frame(const offk_stencil_t& s, int f) {
  const int P = s.B * (s.L - 1);
  if (s.index_mode == OFFK_INDEX_REFERENCE_FLAT) return f < P ? f : -1;
  const int b = f / s.L, t = f - b * s.L;
  return t < s.L - 1 ? b * (s.L - 1) + t : -1;
}
// keep-factors of the 4 spatial outputs (p, och..och+3, pix).  OFFK_DROP_MASK: the mask is indexed like the
// reference's dropout input [P, K*Cs, H, W] (RGB_OFF.py:612), so injected masks keep the reference's layout.
// OFFK_DROP_SEED: one hash per channel quad; quad = channels-last element index ((p*HW + pix)*K*Cs + och) / 4.
__device__ __forceinline__ float4 drop_factor4(const offk_stencil_t& s, uint32_t thr, int p, int och, int pix, int HW,
                                               uint64_t quad) {
  if (s.drop_mode == OFFK_DROP_NONE) return make_float4(1.f, 1.f, 1.f, 1.f);
  uint32_t keep;
  if (s.drop_mode == OFFK_DROP_MASK) {
    const uint8_t* m = s.keep_mask + ((size_t)p * (s.K * s.Cs) + och) * (size_t)HW + pix;
    keep = (m[0] != 0 ? 1u : 0u) | (m[HW] != 0 ? 2u : 0u) | (m[2 * (size_t)HW] != 0 ? 4u : 0u) | (m[3 * (size_t)HW] != 0 ? 8u : 0u);
  } else {
    keep = drop_keep4(s.seed + (s.seed_dev ? __ldg(s.seed_dev) : 0ull), quad, thr);
  }
  const float k = s.keep_scale;
  return make_float4(keep & 1u ? k : 0.f, keep & 2u ? k : 0.f, keep & 4u ? k : 0.f, keep & 8u ? k : 0.f);
}

__device__ __forceinline__ const StLevel& find_level(const StBatch& bt, int blk) {
  int li = 0;
#pragma unroll 1
  while (li + 1 < bt.n && blk >= bt.lv[li + 1].blk0) ++li;
  return bt.lv[li];
}

// Spatial blocks sit at every (1 << lstride)-th position of the level's block range until all are placed; the other
// positions are temporal blocks.  Returns the spatial index (>= 0) or ~temporal index.
__device__ __forceinline__ int block_role(const StLevel& lv, int rel) {
  const int ls = lv.lstride, sidx = rel >> ls;
  if ((rel & ((1 << ls) - 1)) == 0 && sidx < lv.n_sblocks) return sidx;
  const int before = min(lv.n_sblocks, (rel + (1 << ls) - 1) >> ls);
  return ~(rel - before);
}

// per-channel taps and bias as float4 over 4 consecutive channels, fixed stride so that the tap index is an immediate
// offset: ws4[(kk*9 + j)*ST_WQ + c4], bs4[kk*ST_WQ + c4]
__device__ __forceinline__ void load_taps(const StLevel& lv, float4* ws4, float4* bs4, int tid) {
  const int K = lv.s.K, Cs = lv.s.Cs, K9 = K * 9, CQ = 1 << lv.lq;
  for (int i = tid; i < K9 * ST_WQ; i += ST_THREADS) {
    const int c4 = i & (ST_WQ - 1), kj = i / ST_WQ;
    if (c4 < CQ) {
      const float* b = lv.w + (size_t)(c4 * 4) * K9 + kj;          // w[c][kk][3][3]: channel stride K*9
      ws4[i] = make_float4(__ldg(b), __ldg(b + K9), __ldg(b + 2 * K9), __ldg(b + 3 * K9));
    }
  }
  if (bs4) {
    for (int i = tid; i < K * ST_WQ; i += ST_THREADS) {
      const int c4 = i & (ST_WQ - 1), kk = i / ST_WQ;
      if (c4 < CQ) bs4[i] = lv.bias ? ldg4(lv.bias + kk * Cs + c4 * 4) : f4zero();
    }
  }
}

struct StNoXform {
  __device__ __forceinline__ float4 operator()(float4 v, int) const { return v; }
};

// Stage rows [y0-1, y0+rows] x columns [-1, W] x Cs channels of frame `src` into tile[(r*TCP + col)*CQ + c4]
// (zero outside the plane).  RAW: 16-byte cp.async with zero-fill; otherwise through registers with `xform`.
template <bool RAW, typename F>
__device__ __forceinline__ void stage_tile(const StLevel& lv, float4* tile, const float* src, int src_ps, int y0, int rows,
                                           int tid, F xform) {
  const int H = lv.s.H, W = lv.s.W, lq = lv.lq, lcpr = lv.ltcp + lv.lq, CQ = 1 << lq;
  const uint32_t tile_s = st_smem_u32(tile);
  if ((1 << lcpr) <= ST_THREADS) {
    // a thread owns one (column, channel quad) and walks the rows
    const int rr = tid >> lcpr, within = tid & ((1 << lcpr) - 1), col = within >> lq, c4 = within & (CQ - 1);
    const int rpi = ST_THREADS >> lcpr, xx = col - 1;
    const bool colok = col < W + 2, xin = xx >= 0 && xx < W;
    int off = ((y0 - 1 + rr) * W + xx) * src_ps + c4 * 4;
    int cell = (rr << lcpr) + within;
    const int off_step = rpi * W * src_ps, cell_step = rpi << lcpr;
    for (int r = rr; r < rows + 2; r += rpi, off += off_step, cell += cell_step) {
      const int yy = y0 - 1 + r;
      const bool in = xin && yy >= 0 && yy < H;
      if (colok) {
        if (RAW) st_cp_async16(tile_s + (uint32_t)cell * 16u, in ? src + off : src, in ? 16u : 0u);
        else tile[cell] = in ? xform(ldg4(src + off), yy * W + xx) : f4zero();
      }
    }
  } else {
    const int TCP = 1 << lv.ltcp;
    const int n_cells = (rows + 2) << lcpr;
    for (int i = tid; i < n_cells; i += ST_THREADS) {
      const int c4 = i & (CQ - 1), col = (i >> lq) & (TCP - 1), r = i >> lcpr;
      if (col < W + 2) {
        const int yy = y0 - 1 + r, xx = col - 1;
        const bool in = yy >= 0 && yy < H && xx >= 0 && xx < W;
        const int off = (yy * W + xx) * src_ps + c4 * 4;
        if (RAW) st_cp_async16(tile_s + (uint32_t)i * 16u, in ? src + off : src, in ? 16u : 0u);
        else tile[i] = in ? xform(ldg4(src + off), yy * W + xx) : f4zero();
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------- forward
// temporal difference (RGB_OFF.py:599-604).  LT = 3: fully unrolled, the three frames of a pixel pair in flight together;
// LT = 0: any L, frames t+1 and t+2 requested before the difference of frame t is stored.
template <int LT>
__device__ __forceinline__ void temporal_fwd(const StLevel& lv, int r2, int tid) {
  const int L = lv.s.L, Cg = lv.s.Cg, HW = lv.s.H * lv.s.W;
  const size_t g_fs = (size_t)lv.s.g_fs, o_fs = (size_t)HW * lv.s.out_ctot;
  const int g_ps = lv.s.g_ps, ctot = lv.s.out_ctot;
  const int b = r2 / lv.t_chunks, chunk = r2 - b * lv.t_chunks;
  const int warp = tid >> 5, lane = tid & 31;
  const int pixw = chunk * ST_TPIX + warp * (2 * ST_TIT);
  for (int c = lane * 4; c < Cg; c += 128) {
    const float* g0 = lv.g + (size_t)b * L * g_fs + (size_t)pixw * g_ps + c;
    float* o0 = lv.out + (size_t)b * (L - 1) * o_fs + (size_t)pixw * ctot + lv.s.out_coff + lv.s.K * lv.s.Cs + c;
#pragma unroll 1
    for (int it = 0; it < ST_TIT; ++it, g0 += 2 * g_ps, o0 += 2 * ctot) {
      const int pix0 = pixw + it * 2;
      if (pix0 >= HW) break;
      const bool ok1 = pix0 + 1 < HW;                              // the second pixel of the pair may fall off the plane
      const float* gp0 = g0;
      const float* gp1 = ok1 ? g0 + g_ps : g0;                     // clamped: duplicate loads, predicated stores
      float* op0 = o0;
      float* op1 = o0 + ctot;
      if (LT == 3) {
        const float4 a0 = ldg_stream4(gp0), a1 = ldg_stream4(gp1);
        const float4 b0 = ldg_stream4(gp0 + g_fs), b1 = ldg_stream4(gp1 + g_fs);
        const float4 c0 = ldg_stream4(gp0 + 2 * g_fs), c1 = ldg_stream4(gp1 + 2 * g_fs);
        stg_stream4(op0, f4sub(b0, a0));
        if (ok1) stg_stream4(op1, f4sub(b1, a1));
        stg_stream4(op0 + o_fs, f4sub(c0, b0));
        if (ok1) stg_stream4(op1 + o_fs, f4sub(c1, b1));
      } else {
        float4 p0 = ldg_stream4(gp0), p1 = ldg_stream4(gp1);
        gp0 += g_fs; gp1 += g_fs;
        float4 c0 = ldg_stream4(gp0), c1 = ldg_stream4(gp1);
        float4 n0 = f4zero(), n1 = f4zero(), m0 = f4zero(), m1 = f4zero();
        if (L > 2) {
          gp0 += g_fs; gp1 += g_fs;
          n0 = ldg_stream4(gp0); n1 = ldg_stream4(gp1);
        }
        for (int t = 1; t < L; ++t) {
          if (t + 2 < L) {
            gp0 += g_fs; gp1 += g_fs;
            m0 = ldg_stream4(gp0); m1 = ldg_stream4(gp1);
          }
          stg_stream4(op0, f4sub(c0, p0));
          if (ok1) stg_stream4(op1, f4sub(c1, p1));
          op0 += o_fs; op1 += o_fs;
          p0 = c0; p1 = c1; c0 = n0; c1 = n1; n0 = m0; n1 = m1;
        }
      }
    }
  }
}

// spatial gradient (RGB_OFF.py:611 / Flow_OFF.py:622 / util.py:46-50) + bias + dropout for one (pair, band) item
template <int KK>
__device__ __forceinline__ void spatial_fwd(const StLevel& lv, int item, int tid, float4* st_smem) {
  const offk_stencil_t& s = lv.s;
  const int H = s.H, W = s.W, HW = H * W, Cs = s.Cs, ctot = s.out_ctot;
  const int p = item / lv.bands, band = item - p * lv.bands;
  const int y0 = band * lv.band_rows;
  const int rows = min(lv.band_rows, H - y0);
  const int lq = lv.lq, ltcp = lv.ltcp, CQ = 1 << lq;
  float4* tile = st_smem;                                        // [rows+2][TCP][CQ]
  float4* ws4 = st_smem + ((lv.band_rows + 2) << (ltcp + lq));   // [K*9][ST_WQ]
  float4* bs4 = ws4 + KK * 9 * ST_WQ;                            // [K][ST_WQ]
  stage_tile<true>(lv, tile, lv.d + (size_t)spatial_frame(s, p) * s.d_fs, s.d_ps, y0, rows, tid, StNoXform());
  load_taps(lv, ws4, bs4, tid);
  st_cp_async_wait_all();
  __syncthreads();

  const int c4 = tid & (CQ - 1), slot = tid >> lq;
  const int lpw = lv.lpw, PW = (W + 1) >> 1;                     // pixel pairs per row
  const int rpp = (ST_THREADS >> lq) >> lpw;                     // rows per pass
  const int sx = slot & ((1 << lpw) - 1), sy = slot >> lpw;
  const uint32_t thr = drop_threshold16(s.drop_p);
  const float4* wk = ws4 + c4;
  float4 wr[9];
#pragma unroll
  for (int j = 0; j < 9; ++j) wr[j] = wk[j * ST_WQ];             // first map's taps live in registers
  const float4 b0 = bs4[c4], b1 = KK > 1 ? bs4[ST_WQ + c4] : f4zero();
  const int rs = 1 << (ltcp + lq);                               // tile row stride (float4)
  float* obase = lv.out + (size_t)p * HW * ctot + s.out_coff + c4 * 4;
  const uint32_t qbase = (uint32_t)p * (uint32_t)HW;             // dropout: quad index = ((p*HW + pix)*K*Cs + och) / 4
  const uint32_t kcq = (uint32_t)(KK * Cs) >> 2;
  for (int yb = 0; yb < rows; yb += rpp) {
    const int y = yb + sy;
    for (int xp0 = 0; xp0 < PW; xp0 += 1 << lpw) {
      const int x = (xp0 + sx) * 2;
      if (y < rows && x < W) {
        const float4* r0 = tile + (((y << ltcp) + x) << lq) + c4;       // halo coordinates: (y, x) = top-left neighbour
        float4 e0 = b0, e1 = b0, f0 = b1, f1 = b1;                      // e: map 0 at x / x+1, f: map 1
#pragma unroll
        for (int a = 0; a < 3; ++a) {
          const float4* ra = r0 + a * rs;
          const float4 n0 = ra[0], n1 = ra[CQ], n2 = ra[2 * CQ], n3 = ra[3 * CQ];
          f4fma(e0, wr[a * 3], n0); f4fma(e0, wr[a * 3 + 1], n1); f4fma(e0, wr[a * 3 + 2], n2);
          f4fma(e1, wr[a * 3], n1); f4fma(e1, wr[a * 3 + 1], n2); f4fma(e1, wr[a * 3 + 2], n3);
          if (KK > 1) {
            const float4 u0 = wk[(9 + a * 3) * ST_WQ], u1 = wk[(10 + a * 3) * ST_WQ], u2 = wk[(11 + a * 3) * ST_WQ];
            f4fma(f0, u0, n0); f4fma(f0, u1, n1); f4fma(f0, u2, n2);
            f4fma(f1, u0, n1); f4fma(f1, u1, n2); f4fma(f1, u2, n3);
          }
        }
        const int pix = (y0 + y) * W + x;
        float* op = obase + (size_t)pix * ctot;
        const uint64_t q = (uint64_t)(qbase + pix) * kcq + c4;
        stg_stream4(op, f4mul(e0, drop_factor4(s, thr, p, c4 * 4, pix, HW, q)));
        if (KK > 1) stg_stream4(op + Cs, f4mul(f0, drop_factor4(s, thr, p, Cs + c4 * 4, pix, HW, q + (Cs >> 2))));
        if (x + 1 < W) {
          stg_stream4(op + ctot, f4mul(e1, drop_factor4(s, thr, p, c4 * 4, pix + 1, HW, q + kcq)));
          if (KK > 1)
            stg_stream4(op + ctot + Cs, f4mul(f1, drop_factor4(s, thr, p, Cs + c4 * 4, pix + 1, HW, q + kcq + (Cs >> 2))));
        }
      }
    }
  }
}

__global__ void __launch_bounds__(ST_THREADS, ST_FWD_MINB)
stencil_diff_fwd_kernel(const __grid_constant__ StBatch bt) {
  pdl_sync();
  extern __shared__ __align__(16) float4 st_smem[];
  const StLevel& lv = find_level(bt, (int)blockIdx.x);
  const int tid = threadIdx.x;
  const int role = block_role(lv, (int)blockIdx.x - lv.blk0);
  if (role < 0) {
    if (lv.s.L == 3) temporal_fwd<3>(lv, ~role, tid);
    else temporal_fwd<0>(lv, ~role, tid);
  } else {
    if (lv.s.K == 1) spatial_fwd<1>(lv, role, tid, st_smem);
    else spatial_fwd<2>(lv, role, tid, st_smem);
  }
}

// ---------------------------------------------------------------------------------------------- backward
// dG[b,t] = (dT[b,t-1] - dT[b,t]) * (G[b,t] > 0)      (ReLU' of RGB_OFF.py:598): same walk as the forward
template <int LT>
__device__ __forceinline__ void temporal_bwd(const StLevel& lv, int r2, int tid) {
  const int L = lv.s.L, Cg = lv.s.Cg, HW = lv.s.H * lv.s.W;
  const size_t g_fs = (size_t)lv.s.g_fs, dg_fs = (size_t)lv.dg_fs, o_fs = (size_t)HW * lv.s.out_ctot;
  const int g_ps = lv.s.g_ps, ctot = lv.s.out_ctot;
  const int b = r2 / lv.t_chunks, chunk = r2 - b * lv.t_chunks;
  const int warp = tid >> 5, lane = tid & 31;
  const int pixw = chunk * ST_TPIX + warp * (2 * ST_TIT);
  for (int c = lane * 4; c < Cg; c += 128) {
    const float* g0 = lv.g + (size_t)b * L * g_fs + (size_t)pixw * g_ps + c;
    float* d0 = lv.dg + (size_t)b * L * dg_fs + (size_t)pixw * g_ps + c;                 // dg uses the pixel stride of g
    const float* o0 = lv.dout + (size_t)b * (L - 1) * o_fs + (size_t)pixw * ctot + lv.s.out_coff + lv.s.K * lv.s.Cs + c;
#pragma unroll 1
    for (int it = 0; it < ST_TIT; ++it, g0 += 2 * g_ps, d0 += 2 * g_ps, o0 += 2 * ctot) {
      const int pix0 = pixw + it * 2;
      if (pix0 >= HW) break;
      const bool ok1 = pix0 + 1 < HW;
      const float* gp0 = g0;
      const float* gp1 = ok1 ? g0 + g_ps : g0;
      const float* op0 = o0;
      const float* op1 = ok1 ? o0 + ctot : o0;
      float* dp0 = d0;
      float* dp1 = d0 + g_ps;
      if (LT == 3) {
        const float4 ga0 = ldg_stream4(gp0), ga1 = ldg_stream4(gp1);
        const float4 ta0 = ldg_stream4(op0), ta1 = ldg_stream4(op1);
        const float4 gb0 = ldg_stream4(gp0 + g_fs), gb1 = ldg_stream4(gp1 + g_fs);
        const float4 tb0 = ldg_stream4(op0 + o_fs), tb1 = ldg_stream4(op1 + o_fs);
        const float4 gc0 = ldg_stream4(gp0 + 2 * g_fs), gc1 = ldg_stream4(gp1 + 2 * g_fs);
        stg_stream4(dp0, relu_gate4(ga0, f4sub(f4zero(), ta0)));
        if (ok1) stg_stream4(dp1, relu_gate4(ga1, f4sub(f4zero(), ta1)));
        stg_stream4(dp0 + dg_fs, relu_gate4(gb0, f4sub(ta0, tb0)));
        if (ok1) stg_stream4(dp1 + dg_fs, relu_gate4(gb1, f4sub(ta1, tb1)));
        stg_stream4(dp0 + 2 * dg_fs, relu_gate4(gc0, tb0));
        if (ok1) stg_stream4(dp1 + 2 * dg_fs, relu_gate4(gc1, tb1));
      } else {
        float4 pv0 = f4zero(), pv1 = f4zero();
        float4 gv0 = ldg_stream4(gp0), gv1 = ldg_stream4(gp1);
        float4 dt0 = ldg_stream4(op0), dt1 = ldg_stream4(op1);     // L >= 2: pair 0 exists
        float4 ng0 = f4zero(), ng1 = f4zero(), nd0, nd1;
        for (int t = 0; t < L; ++t) {
          if (t + 1 < L) {
            gp0 += g_fs; gp1 += g_fs;
            ng0 = ldg_stream4(gp0); ng1 = ldg_stream4(gp1);
          }
          nd0 = f4zero(); nd1 = f4zero();
          if (t + 1 < L - 1) {
            op0 += o_fs; op1 += o_fs;
            nd0 = ldg_stream4(op0); nd1 = ldg_stream4(op1);
          }
          stg_stream4(dp0, relu_gate4(gv0, f4sub(pv0, dt0)));
          if (ok1) stg_stream4(dp1, relu_gate4(gv1, f4sub(pv1, dt1)));
          dp0 += dg_fs; dp1 += dg_fs;
          pv0 = dt0; pv1 = dt1; dt0 = nd0; dt1 = nd1; gv0 = ng0; gv1 = ng1;
        }
      }
    }
  }
}

// spatial blocks: dD = transposed stencil of the dropped dS; tap / bias gradients.  A block owns `ipb` consecutive
// (frame, band) items and keeps the tap-gradient partial sums in registers across them.  Per item, the dS band + halo
// and the D band are staged with 16-byte cp.async (everything in flight at once: one exposed memory latency per
// item), dropout' is applied to the staged tile in place, and the compute passes touch shared memory only.
__device__ __forceinline__ void spatial_bwd(const StLevel& lv, int rel, int tid, float4* st_smem) {
  const offk_stencil_t& s = lv.s;
  const int H = s.H, W = s.W, HW = H * W, K = s.K, Cs = s.Cs, ctot = s.out_ctot, d_ps = s.d_ps;
  const int lq = lv.lq, ltcp = lv.ltcp, CQ = 1 << lq, lcpr = ltcp + lq;
  float4* tile = st_smem;                                        // dS band + halo [rows+2][TCP][CQ]
  float4* dband = st_smem + ((lv.band_rows + 2) << lcpr);        // D band [rows][W][CQ]
  const bool need_dw = lv.dw != nullptr, need_db = lv.dbias != nullptr;
  const bool need_acc = need_dw || need_db;
  float4* ws4 = dband + (need_dw ? (lv.band_rows * W) << lq : 0);   // [K*9][ST_WQ]  (the D band exists only with dw)
  float* redw = reinterpret_cast<float*>(ws4 + K * 9 * ST_WQ);   // [ST_WARPS][10][Cs] per-warp tap-gradient partials
  bool taps_loaded = false;                                      // loaded under the first item's cp.async traffic
  const int c4 = tid & (CQ - 1), slot = tid >> lq;
  const int XW = 1 << lv.lxw;
  const int rpp = (ST_THREADS >> lq) >> lv.lxw;
  const int sx = slot & (XW - 1), sy = slot >> lv.lxw;
  const int rs = 1 << lcpr;
  const int item0 = rel * lv.ipb, item1 = min(item0 + lv.ipb, lv.n_sitems);
  const uint32_t thr = drop_threshold16(s.drop_p), kcq = (uint32_t)(K * Cs) >> 2;
  const uint32_t dband_s = st_smem_u32(dband);

  for (int kk = 0; kk < K; ++kk) {
    float4 wacc[9], bacc = f4zero();
#pragma unroll
    for (int j = 0; j < 9; ++j) wacc[j] = f4zero();
    const int och = kk * Cs + c4 * 4;
    const float4* wk = ws4 + kk * 9 * ST_WQ + c4;
    bool any_pair = false;
    for (int item = item0; item < item1; ++item) {
      const int f = item / lv.bands, band = item - f * lv.bands;
      const int y0 = band * lv.band_rows;
      const int rows = min(lv.band_rows, H - y0);
      const int p = spatial_pair_of_frame(s, f);
      float* ddf = lv.dd + (size_t)f * lv.dd_fs + c4 * 4;          // dd uses the pixel stride of d
      __syncthreads();                                           // previous item's tiles fully consumed (and ws4 ready)
      if (p < 0) {                                               // frame feeds no pair: dD = 0 (first map only writes)
        if (kk == 0)
          for (int i = slot; i < rows * W; i += ST_THREADS >> lq)
            *reinterpret_cast<float4*>(ddf + (size_t)(y0 * W + i) * d_ps) = f4zero();
        continue;
      }
      any_pair = true;
      const bool use_d = need_dw;
      stage_tile<true>(lv, tile, lv.dout + (size_t)p * HW * ctot + s.out_coff + kk * Cs, ctot, y0, rows, tid, StNoXform());
      if (use_d) {
        const float* dsrc = lv.d + (size_t)spatial_frame(s, p) * s.d_fs + (size_t)(y0 * W) * d_ps + c4 * 4;
        for (int i = slot; i < rows * W; i += ST_THREADS >> lq)
          st_cp_async16(dband_s + (uint32_t)((i << lq) + c4) * 16u, dsrc + (size_t)i * d_ps, 16u);
      }
      if (!taps_loaded) {
        load_taps(lv, ws4, nullptr, tid);
        taps_loaded = true;
      }
      st_cp_async_wait_all();
      if (s.drop_mode != OFFK_DROP_NONE) {
        // dropout' in place on the landed tile: cell i = tid + k*ST_THREADS is exactly the set of cells this thread
        // staged itself (stage_tile's three index walks all reduce to it), so its own wait_group is enough -- no barrier
        const int n_cells = (rows + 2) << lcpr;
        const uint32_t qbase = (uint32_t)p * (uint32_t)HW;
        for (int i = tid; i < n_cells; i += ST_THREADS) {         // ST_THREADS % CQ == 0: i & (CQ-1) == c4
          const int col = (i >> lq) & ((1 << ltcp) - 1), r = i >> lcpr;
          const int yy = y0 - 1 + r, xx = col - 1;
          if (yy >= 0 && yy < H && xx >= 0 && xx < W) {
            const int pix = yy * W + xx;
            tile[i] = f4mul(tile[i], drop_factor4(s, thr, p, och, pix, HW, (uint64_t)(qbase + pix) * kcq + (och >> 2)));
          }
        }
      }
      __syncthreads();
      for (int yb = 0; yb < rows; yb += rpp) {
        const int y = yb + sy;
        for (int x0 = 0; x0 < W; x0 += XW) {
          const int x = x0 + sx;
          if (y < rows && x < W) {
            const int pix = (y0 + y) * W + x;
            float4 acc = f4zero();
            float4 dv = f4zero();
            if (use_d) dv = dband[((y * W + x) << lq) + c4];
            // dS(y-a+1, x-b+1) sits at halo coordinates (y+2-a, x+2-b)
            const float4* t2 = tile + ((((y + 2) << ltcp) + x + 2) << lq) + c4;
#pragma unroll
            for (int a = 0; a < 3; ++a) {
              const float4* ra = t2 - a * rs;
#pragma unroll
              for (int bb = 0; bb < 3; ++bb) {
                const float4 nv = *(ra - bb * CQ);
                f4fma(acc, wk[(a * 3 + bb) * ST_WQ], nv);
                f4fma(wacc[a * 3 + bb], dv, nv);
                if (a == 1 && bb == 1) { bacc.x += nv.x; bacc.y += nv.y; bacc.z += nv.z; bacc.w += nv.w; }
              }
            }
            float4* o = reinterpret_cast<float4*>(ddf + (size_t)pix * d_ps);
            if (kk > 0) {
              const float4 old = *o;
              acc.x += old.x; acc.y += old.y; acc.z += old.z; acc.w += old.w;
            }
            *o = acc;
          }
        }
      }
    }
    if (need_acc && any_pair) {                                  // block-uniform: items are per block
      // lanes l, l^CQ, l^2CQ, ... hold the same channels: butterfly over them, then one slot per warp (no atomics)
      const int warp = tid >> 5, lane = tid & 31;
      float vals[40];
#pragma unroll
      for (int j = 0; j < 9; ++j) { vals[4 * j] = wacc[j].x; vals[4 * j + 1] = wacc[j].y; vals[4 * j + 2] = wacc[j].z; vals[4 * j + 3] = wacc[j].w; }
      vals[36] = bacc.x; vals[37] = bacc.y; vals[38] = bacc.z; vals[39] = bacc.w;
      float* mine = redw + (size_t)warp * 10 * Cs + c4 * 4;
      if (lq == 3) {                                             // Cs = 32 (every OFF unit): two butterfly steps, unrolled
#pragma unroll
        for (int q = 0; q < 40; ++q) {
          float v = vals[q];
          v += __shfl_xor_sync(0xffffffffu, v, 16);
          v += __shfl_xor_sync(0xffffffffu, v, 8);
          vals[q] = v;
        }
      } else {
#pragma unroll
        for (int q = 0; q < 40; ++q) {
          float v = vals[q];
          for (int o = 16; o >= CQ; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
          vals[q] = v;
        }
      }
      if (lane < CQ) {
#pragma unroll
        for (int j = 0; j < 10; ++j)
          *reinterpret_cast<float4*>(mine + j * Cs) = make_float4(vals[4 * j], vals[4 * j + 1], vals[4 * j + 2], vals[4 * j + 3]);
      }
      __syncthreads();
      for (int i = tid; i < 10 * Cs; i += ST_THREADS) {
        const int j = i / Cs, c = i - j * Cs;
        float v = 0.f;
#pragma unroll
        for (int w8 = 0; w8 < ST_WARPS; ++w8) v += redw[w8 * 10 * Cs + i];
        if (j < 9) {
          if (need_dw) atomicAdd(lv.dw + ((size_t)c * K + kk) * 9 + j, v);
        } else if (need_db) {
          atomicAdd(lv.dbias + kk * Cs + c, v);
        }
      }
    }
  }
}

__global__ void __launch_bounds__(ST_THREADS, ST_FWD_MINB)
stencil_diff_bwd_kernel(const __grid_constant__ StBatch bt) {
  pdl_sync();
  extern __shared__ __align__(16) float4 st_smem[];
  const StLevel& lv = find_level(bt, (int)blockIdx.x);
  const int tid = threadIdx.x;
  const int role = block_role(lv, (int)blockIdx.x - lv.blk0);
  if (role < 0) {
    if (lv.s.L == 3) temporal_bwd<3>(lv, ~role, tid);
    else temporal_bwd<0>(lv, ~role, tid);
  } else {
    spatial_bwd(lv, role, tid, st_smem);
  }
}

// ---------------------------------------------------------------------------------------------- host
static int check_stencil(const offk_stencil_t* s) {
  OFFK_REQUIRE(s != nullptr, "stencil: null descriptor");
  OFFK_REQUIRE(s->B >= 1 && s->L >= 2, "stencil: need B >= 1 and L >= 2 (got B=%d L=%d)", s->B, s->L);
  OFFK_REQUIRE(s->Cg >= 0 && s->Cs >= 0 && s->Cg + s->Cs > 0, "stencil: bad channel counts");
  OFFK_REQUIRE(s->Cg % 4 == 0 && s->Cs % 4 == 0 && s->Cs <= ST_MAX_CS, "stencil: channels must be multiples of 4, Cs <= %d",
               ST_MAX_CS);
  OFFK_REQUIRE(s->Cs == 0 || (((s->Cs >> 2) & ((s->Cs >> 2) - 1)) == 0), "stencil: Cs/4 must be a power of two");
  OFFK_REQUIRE(s->H >= 1 && s->W >= 1 && s->H < 32768 && s->W < 32768, "stencil: plane size");
  OFFK_REQUIRE(s->K >= 1 && s->K <= 2, "stencil: K must be 1 or 2");
  OFFK_REQUIRE(s->out_coff >= 0 && s->out_coff + s->K * s->Cs + s->Cg <= s->out_ctot, "stencil: channel slice");
  OFFK_REQUIRE(s->out_ctot % 4 == 0 && s->out_coff % 4 == 0, "stencil: output slice must be float4-aligned");
  OFFK_REQUIRE(s->g_fs % 4 == 0 && s->d_fs % 4 == 0 && s->g_ps % 4 == 0 && s->d_ps % 4 == 0, "stencil: strides");
  OFFK_REQUIRE(s->drop_mode >= 0 && s->drop_mode <= 2, "stencil: drop_mode");
  OFFK_REQUIRE(s->drop_mode != OFFK_DROP_MASK || s->keep_mask, "stencil: OFFK_DROP_MASK needs keep_mask");
  return 0;
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
static int ilog2_ceil(int v) {
  int l = 0;
  while ((1 << l) < v) ++l;
  return l;
}

// geometry of the spatial blocks of one level; returns the dynamic shared memory the level needs (0 if Cs == 0)
static int plan_spatial(StLevel& lv, bool backward) {
  const offk_stencil_t& s = lv.s;
  lv.lq = lv.ltcp = lv.lxw = lv.lpw = 0;
  lv.ipb = 1;
  lv.bands = lv.band_rows = 1;
  lv.n_sitems = lv.n_sblocks = 0;
  if (s.Cs == 0) return 0;
  const int CQ = s.Cs / 4;
  lv.lq = ilog2_ceil(CQ);
  lv.ltcp = ilog2_ceil(s.W + 2);
  const int row_bytes = (1 << lv.ltcp) * CQ * 16;
  int max_rows = ST_TILE_BUDGET / row_bytes - 2;
  if (max_rows < 1) max_rows = 1;
  lv.bands = (s.H + max_rows - 1) / max_rows;
  lv.band_rows = (s.H + lv.bands - 1) / lv.bands;
  lv.bands = (s.H + lv.band_rows - 1) / lv.band_rows;
  const int slots = ST_THREADS / CQ;
  int lxw = ilog2_ceil(s.W);
  while ((1 << lxw) > slots) --lxw;
  lv.lxw = lxw;
  int lpw = ilog2_ceil((s.W + 1) / 2);
  while ((1 << lpw) > slots) --lpw;
  lv.lpw = lpw;
  const long long units = backward ? (long long)s.B * s.L : (long long)s.B * (s.L - 1);
  const long long items = units * lv.bands;
  lv.n_sitems = (int)items;
  // backward: a block keeps the tap-gradient partial sums in registers over up to ST_ITEMS consecutive items (fewer
  // block reductions / atomics); small levels keep one item per block so their blocks stay short
  // measured at config 2 (B200): items / (0.5 * SMs) capped at 8 -> 121 us; 2.0 / 4 -> 149 us; 0.2 / 32 -> 250 us (tail)
  const long long ipb = items * 2 / sm_count();
  lv.ipb = backward ? (int)(ipb < 1 ? 1 : (ipb > ST_ITEMS ? ST_ITEMS : ipb)) : 1;
  lv.n_sblocks = (int)((items + lv.ipb - 1) / lv.ipb);
  const int tile_bytes = (lv.band_rows + 2) * row_bytes;
  const int tap_bytes = s.K * 9 * ST_WQ * 16;
  // backward: + the D band (no halo) and one tap-gradient partial slot per warp
  const int extra = backward ? (lv.dw ? lv.band_rows * s.W * CQ * 16 : 0) + ((lv.dw || lv.dbias) ? ST_WARPS * 10 * s.Cs * 4 : 0)
                             : s.K * ST_WQ * 16;
  return tile_bytes + tap_bytes + extra;
}

static int launch_batch(int n, const offk_stencil_t* s, const offk_stencil_io_t* io, bool backward, void* stream) {
  OFFK_REQUIRE(n >= 1 && n <= ST_MAX_LEVELS, "stencil batch: 1 <= n <= %d (got %d)", ST_MAX_LEVELS, n);
  OFFK_REQUIRE(s != nullptr && io != nullptr, "stencil batch: null arrays");
  StBatch bt;
  bt.n = n;
  long long blk = 0;
  int smem = 0;
  for (int i = 0; i < n; ++i) {
    if (int e = check_stencil(&s[i])) return e;
    StLevel& lv = bt.lv[i];
    lv.s = s[i];
    lv.g = io[i].g; lv.d = io[i].d; lv.w = io[i].w; lv.bias = io[i].bias; lv.out = io[i].out;
    lv.dout = io[i].dout; lv.dg = io[i].dg; lv.dd = io[i].dd; lv.dw = io[i].dw; lv.dbias = io[i].dbias;
    lv.dg_fs = io[i].dg_fs; lv.dd_fs = io[i].dd_fs;
    if (!backward) {
      OFFK_REQUIRE(lv.out != nullptr && aligned16(lv.out), "stencil_fwd: out must be non-null and 16-byte aligned");
      OFFK_REQUIRE(s[i].Cg == 0 || (lv.g && aligned16(lv.g)), "stencil_fwd: g must be 16-byte aligned");
      OFFK_REQUIRE(s[i].Cs == 0 || (lv.d && lv.w && aligned16(lv.d)), "stencil_fwd: d / w missing or unaligned");
      OFFK_REQUIRE(lv.bias == nullptr || aligned16(lv.bias), "stencil_fwd: bias must be 16-byte aligned");
    } else {
      OFFK_REQUIRE(lv.dout != nullptr && aligned16(lv.dout), "stencil_bwd: dout must be 16-byte aligned");
      OFFK_REQUIRE(s[i].Cg == 0 || (lv.g && lv.dg && aligned16(lv.g) && aligned16(lv.dg) && lv.dg_fs % 4 == 0), "stencil_bwd: g/dg");
      OFFK_REQUIRE(s[i].Cs == 0 || (lv.w && lv.dd && aligned16(lv.dd) && lv.dd_fs % 4 == 0), "stencil_bwd: w/dd missing");
      OFFK_REQUIRE(lv.dw == nullptr || (lv.d != nullptr && aligned16(lv.d)), "stencil_bwd: tap gradient needs d");
    }
    const int need = plan_spatial(lv, backward);
    OFFK_REQUIRE(need <= ST_SMEM_MAX, "stencil: halo tile of %d bytes exceeds %d (W=%d, Cs=%d)", need, ST_SMEM_MAX, s[i].W, s[i].Cs);
    if (need > smem) smem = need;
    const int HW = s[i].H * s[i].W;
    lv.t_chunks = s[i].Cg > 0 ? (HW + ST_TPIX - 1) / ST_TPIX : 1;
    const long long n_t = s[i].Cg > 0 ? (long long)lv.t_chunks * s[i].B : 0;
    lv.n_tblocks = (int)n_t;
    // spatial blocks at every 2^lstride-th position of the level's range
    lv.lstride = 0;
    if (lv.n_sblocks > 0)
      while (((long long)lv.n_sblocks << (lv.lstride + 1)) <= lv.n_sblocks + n_t) ++lv.lstride;
    lv.blk0 = (int)blk;
    blk += lv.n_sblocks + n_t;
    OFFK_REQUIRE(blk < 2147483647LL, "stencil: grid too large");
  }
  if (blk == 0) return 0;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(stencil_diff_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ST_SMEM_MAX);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(stencil_diff_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ST_SMEM_MAX);
    if (e != cudaSuccess) return cuda_check(e, "cudaFuncSetAttribute(stencil)");
    attr_set = true;
  }
  if (!backward) {
    (void)launch_pdl(stencil_diff_fwd_kernel, dim3((unsigned)blk), dim3(ST_THREADS), (size_t)smem, as_stream(stream), bt);
    return OFFK_LAUNCH_CHECK("stencil_diff_fwd");
  }
  (void)launch_pdl(stencil_diff_bwd_kernel, dim3((unsigned)blk), dim3(ST_THREADS), (size_t)smem, as_stream(stream), bt);
  return OFFK_LAUNCH_CHECK("stencil_diff_bwd");
}

}  // namespace offk

using namespace offk;

extern "C" int offk_stencil_diff_fwd_batch(int n, const offk_stencil_t* s, const offk_stencil_io_t* io, void* stream) {
  return launch_batch(n, s, io, false, stream);
}

extern "C" int offk_stencil_diff_bwd_batch(int n, const offk_stencil_t* s, const offk_stencil_io_t* io, void* stream) {
  return launch_batch(n, s, io, true, stream);
}

extern "C" int offk_stencil_diff_fwd(const offk_stencil_t* s, const float* g, const float* d, const float* w,
                                     const float* bias, float* out, void* stream) {
  offk_stencil_io_t io = {};
  io.g = g; io.d = d; io.w = w; io.bias = bias; io.out = out;
  return launch_batch(1, s, &io, false, stream);
}

extern "C" int offk_stencil_diff_bwd(const offk_stencil_t* s, const float* dout, const float* g, const float* d,
                                     const float* w, float* dg, int64_t dg_fs, float* dd, int64_t dd_fs, float* dw,
                                     float* dbias, void* stream) {
  offk_stencil_io_t io = {};
  io.g = g; io.d = d; io.w = w; io.dout = dout; io.dg = dg; io.dg_fs = dg_fs; io.dd = dd; io.dd_fs = dd_fs;
  io.dw = dw; io.dbias = dbias;
  return launch_batch(1, s, &io, true, stream);
}
