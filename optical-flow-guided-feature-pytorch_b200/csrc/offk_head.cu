// Head-side kernels of the OFF sub-network (channels-last tensors [P, HW, C]): global average pool (+dropout) forward/backward,
// the channels-last 3x3 pools (also those of the BN-Inception extractor), the image conversion of the extractor, segment consensus (mean over segments) and small element-wise passes.
// All are bandwidth-trivial ([P,C,7,7] tensors); they exist so that no ATen op is left on the path.
#include "offk_common.cuh"

namespace offk {

__device__ __forceinline__ float keep_factor(int mode, const uint8_t* mask, uint64_t seed, uint32_t thr, size_t idx,
                                             float scale) {
  if (mode == OFFK_DROP_NONE) return 1.f;
  const bool keep = mode == OFFK_DROP_MASK ? (mask[idx] != 0) : drop_keep(seed, idx, thr);
  return keep ? scale : 0.f;
}

// the per-step word of the dropout seed lives in device memory (offk.h: seed_dev)
__global__ void seed_update_kernel(uint64_t* state, uint64_t value) {
  pdl_sync();
  *state = value;
}

// thread per (p, c); x is channels-last [P, HW, ctot]: consecutive threads read consecutive channels
__global__ void avgpool_drop_fwd_kernel(const float* __restrict__ x, int P, int C, int HW, int ctot, int coff, int mode,
                                        const uint8_t* __restrict__ mask, uint64_t seed, const uint64_t* __restrict__ seed_dev,
                                        float drop_p, float scale, float* __restrict__ out) {
  pdl_sync();
  if (seed_dev) seed += __ldg(seed_dev);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P * C) return;
  const int p = i / C, c = i - p * C;
  const float* xp = x + (size_t)p * HW * ctot + coff + c;
  float s = 0.f;
  for (int h = 0; h < HW; ++h) s += __ldg(xp + (size_t)h * ctot);
  const float k = keep_factor(mode, mask, seed, drop_threshold16(drop_p), (size_t)i, scale);
  out[i] = (s / (float)HW) * k;
}

// 3x3 pool over a channel slice of a channels-last tensor, ceil-mode output, one thread per (output pixel, channel quad):
// kind 0 = max over the valid window elements (F.max_pool2d), 1 = sum / 9 (F.avg_pool2d, count_include_pad=True, for
// windows that stay inside the padded input -- every pool the plans use)
__global__ void __launch_bounds__(256) pool3_nhwc_kernel(const float* __restrict__ x, int H, int W, int x_ctot, int x_coff,
                                                         int CQ, int stride, int pad, int kind, int Ho, int Wo, long long total,
                                                         float* __restrict__ y, int y_ctot, int y_coff) {
  pdl_sync();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int cq = (int)(i % CQ);
  const long long pix = i / CQ;                   // (img * Ho + oh) * Wo + ow
  const int ow = (int)(pix % Wo);
  const int oh = (int)((pix / Wo) % Ho);
  const long long img = pix / ((long long)Wo * Ho);
  const float* xp = x + img * H * W * (long long)x_ctot + x_coff + 4 * cq;
  const int y0 = oh * stride - pad, x0 = ow * stride - pad;
  float4 m = kind == 0 ? make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const int yy = y0 + a;
    if (yy < 0 || yy >= H) continue;
#pragma unroll
    for (int b = 0; b < 3; ++b) {
      const int xx = x0 + b;
      if (xx < 0 || xx >= W) continue;
      const float4 v = __ldg(reinterpret_cast<const float4*>(xp + (long long)(yy * W + xx) * x_ctot));
      if (kind == 0) {
        m.x = fmaxf(m.x, v.x); m.y = fmaxf(m.y, v.y); m.z = fmaxf(m.z, v.z); m.w = fmaxf(m.w, v.w);
      } else {
        m.x += v.x; m.y += v.y; m.z += v.z; m.w += v.w;
      }
    }
  }
  if (kind != 0) {
    m.x /= 9.f; m.y /= 9.f; m.z /= 9.f; m.w /= 9.f;
  }
  *reinterpret_cast<float4*>(y + pix * y_ctot + y_coff + 4 * cq) = m;
}

// NCHW image batch [n, c, hw] -> channels-last [n, hw, c_pad], channels >= c zero: one thread per pixel, the c reads are
// coalesced across the warp, the c_pad / 4 float4 stores are contiguous per thread
__global__ void __launch_bounds__(256) image_to_nhwc_kernel(const float* __restrict__ src, float* __restrict__ dst, int c, int hw,
                                                            int c_pad, long long total) {
  pdl_sync();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long img = i / hw;
  const int p = (int)(i - img * hw);
  const float* s = src + img * c * (long long)hw + p;
  float* d = dst + i * c_pad;
  for (int q = 0; q < c_pad; q += 4) {
    float4 v;
    v.x = q + 0 < c ? __ldg(s + (long long)(q + 0) * hw) : 0.f;
    v.y = q + 1 < c ? __ldg(s + (long long)(q + 1) * hw) : 0.f;
    v.z = q + 2 < c ? __ldg(s + (long long)(q + 2) * hw) : 0.f;
    v.w = q + 3 < c ? __ldg(s + (long long)(q + 3) * hw) : 0.f;
    *reinterpret_cast<float4*>(d + q) = v;
  }
}

// ---------------------------------------------------------------------------- fused heads (SURVEY K6)
// One block per output row group: the T frame pairs of one clip when the segment consensus is fused (Flow / v2), else one
// pair (T = 1).  Per pair: global average pool over the HW pixels of the channel slice (consecutive threads = consecutive
// channels: coalesced) + dropout -> shared memory (and `pooled`, which the weight gradient needs) -> 101 x C GEMV by warps
// (float4 along the contiguous weight rows, warp-shuffle reduction) + bias.  Everything is linear, so it is exact fp32 in
// every precision mode.  avgpool -> dropout -> Linear (-> mean over segments): RGB_OFF.py:783-793,844-847; Flow_OFF.py:867-876.
constexpr int HEAD_THREADS = 1024;
constexpr int HEAD_MAX_C = 1024;
constexpr int HEAD_HW_GROUPS = 4;      // pool: the HW pixels of a channel quad are split over 4 thread groups

// All three head kernels are latency-bound (a few hundred KB per block, ~100 blocks): they are written so that every thread
// has its loads in flight together (fully unrolled batches) instead of walking a long dependent loop.
__global__ void __launch_bounds__(HEAD_THREADS) head_fwd_kernel(const float* __restrict__ x, int C, int HW, int ctot, int coff,
                                                                 int mode, const uint8_t* __restrict__ mask, uint64_t seed,
                                                                 const uint64_t* __restrict__ seed_dev, float drop_p, float scale,
                                                                 const float* __restrict__ W, const float* __restrict__ bias,
                                                                 int NC, int T, float* __restrict__ pooled,
                                                                 float* __restrict__ out, float* __restrict__ cout) {
  __shared__ __align__(16) float sp[HEAD_MAX_C];
  __shared__ __align__(16) float spart[HEAD_HW_GROUPS - 1][HEAD_MAX_C];
  pdl_sync();
  if (seed_dev) seed += __ldg(seed_dev);
  const uint32_t thr = drop_threshold16(drop_p);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const float inv_hw = 1.f / (float)HW;
  const int nq = C >> 2;                                         // channel quads (<= 256)
  for (int t = 0; t < T; ++t) {
    const int p = blockIdx.x * T + t;
    const float* xp = x + (size_t)p * HW * ctot + coff;
    // pool: thread = (pixel group hg, channel quad q): pixels hg, hg + 4, ... of quad q, all loads independent
    {
      const int hg = tid / nq, q = tid - hg * nq;
      float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
      if (hg < HEAD_HW_GROUPS) {
#pragma unroll 13
        for (int h = hg; h < HW; h += HEAD_HW_GROUPS) {
          const float4 v = __ldg(reinterpret_cast<const float4*>(xp + (size_t)h * ctot) + q);
          a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
        }
        if (hg > 0) *reinterpret_cast<float4*>(&spart[hg - 1][4 * q]) = a;
      }
      __syncthreads();
      if (hg == 0) {
#pragma unroll
        for (int k = 0; k < HEAD_HW_GROUPS - 1; ++k) {
          const float4 v = *reinterpret_cast<const float4*>(&spart[k][4 * q]);
          a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
        }
        const size_t i0 = (size_t)p * C + 4 * q;
        a.x *= inv_hw * keep_factor(mode, mask, seed, thr, i0, scale);
        a.y *= inv_hw * keep_factor(mode, mask, seed, thr, i0 + 1, scale);
        a.z *= inv_hw * keep_factor(mode, mask, seed, thr, i0 + 2, scale);
        a.w *= inv_hw * keep_factor(mode, mask, seed, thr, i0 + 3, scale);
        *reinterpret_cast<float4*>(sp + 4 * q) = a;
        if (pooled) *reinterpret_cast<float4*>(pooled + i0) = a;
      }
    }
    __syncthreads();
    // Linear: each warp owns up to 4 class rows (n = warp, warp + 32, ...) and walks them TOGETHER along c, so that four
    // independent 16-byte weight loads per lane are in flight per step; warp-shuffle reductions at the end
    {
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
      for (int c = 4 * lane; c < C; c += 128) {
        const float4 p4 = *reinterpret_cast<const float4*>(sp + c);
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const int n = warp + 32 * r;
          if (n < NC) {
            const float4 w4 = __ldg(reinterpret_cast<const float4*>(W + (size_t)n * C + c));
            acc[r] += w4.x * p4.x + w4.y * p4.y + w4.z * p4.z + w4.w * p4.w;
          }
        }
      }
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int n = warp + 32 * r;
        const float v = warp_sum(acc[r]);
        if (lane == 0 && n < NC) out[(size_t)p * NC + n] = v + __ldg(bias + n);
      }
    }
    __syncthreads();
  }
  if (cout) {      // ConsensusModule('avg'): mean over the T rows this block has just written (basic_ops.py:21-22)
    for (int n = tid; n < NC; n += HEAD_THREADS) {
      float s = 0.f;
      for (int t = 0; t < T; ++t) s += out[((size_t)blockIdx.x * T + t) * NC + n];
      cout[(size_t)blockIdx.x * NC + n] = s / (float)T;
    }
  }
}

// dfc(p, n) = dout[(p / T) * NC + n] / T: the consensus backward (basic_ops.py:30-31) folded into the consumers (T = 1: as is)
// dW[n, c] += sum_p dfc(p, n) * pooled[p, c];  db[n] += sum_p dfc(p, n).   block (128 c, 8 n), grid.z cuts the pair axis into
// chunks of HEAD_WG_PAIRS so that the whole machine works on it; partial sums are added with RED.
constexpr int HEAD_WG_PAIRS = 16;
__global__ void __launch_bounds__(1024) head_wgrad_kernel(const float* __restrict__ dout, const float* __restrict__ pooled, int P,
                                                          int C, int NC, int T, float* __restrict__ dW, float* __restrict__ db) {
  pdl_sync();
  const int c = blockIdx.x * 128 + threadIdx.x, n = blockIdx.y * 8 + threadIdx.y;
  if (n >= NC || c >= C) return;
  const int p0 = blockIdx.z * HEAD_WG_PAIRS, p1 = min(P, p0 + HEAD_WG_PAIRS);
  const float invT = 1.f / (float)T;
  float acc = 0.f, accb = 0.f;
#pragma unroll
  for (int i = 0; i < HEAD_WG_PAIRS; ++i) {
    const int p = p0 + i;
    if (p < p1) {
      const float g = __ldg(dout + (size_t)(p / T) * NC + n) * invT;
      acc += g * __ldg(pooled + (size_t)p * C + c);
      accb += g;
    }
  }
  red_add_f32(dW + (size_t)n * C + c, acc);
  if (blockIdx.x == 0 && threadIdx.x == 0 && db) red_add_f32(db + n, accb);
}

// dpool[c] = drop'( sum_n dfc(p, n) * W[n, c] ) / HW, then dx[p, hw, coff + c] = gate( dx_in + dpool[c] ) for every pixel:
// the Linear's data gradient and the average pool's backward (+ the ReLU' of the producer) in one pass.
// Block = (pair p, 256 channels) x 4 class groups: thread (c, ng) sums the classes n = ng, ng + 4, ... (26 independent loads),
// the four partial sums meet in shared memory; then the block's 256 channels x HW pixels go out as float4 stores.
constexpr int HEAD_DG_CH = 256;
constexpr int HEAD_DG_NG = 4;
__global__ void __launch_bounds__(HEAD_DG_CH * HEAD_DG_NG) head_dgrad_kernel(const float* __restrict__ dout, const float* __restrict__ W,
                                                                      int C, int HW, int ctot, int coff, int NC, int T, int mode,
                                                                      const uint8_t* __restrict__ mask, uint64_t seed,
                                                                      const uint64_t* __restrict__ seed_dev, float drop_p,
                                                                      float scale, const float* __restrict__ act, int accumulate,
                                                                      float* __restrict__ dx) {
  __shared__ __align__(16) float sd[HEAD_DG_NG][HEAD_DG_CH];
  __shared__ float sg[128];
  pdl_sync();
  if (seed_dev) seed += __ldg(seed_dev);
  const uint32_t thr = drop_threshold16(drop_p);
  const int tid = threadIdx.x, p = blockIdx.x, c0 = blockIdx.y * HEAD_DG_CH;
  const int cw = min(HEAD_DG_CH, C - c0);                        // channels of this block (a multiple of 4)
  const int cl = tid & (HEAD_DG_CH - 1), ng = tid / HEAD_DG_CH;
  const float invT = 1.f / (float)T;
  for (int n = tid; n < NC; n += HEAD_DG_CH * HEAD_DG_NG) sg[n] = __ldg(dout + (size_t)(p / T) * NC + n) * invT;
  __syncthreads();
  {
    float s = 0.f;
    if (cl < cw) {
      const float* wc = W + c0 + cl;
#pragma unroll 13
      for (int n = ng; n < NC; n += HEAD_DG_NG) s += sg[n] * __ldg(wc + (size_t)n * C);
    }
    sd[ng][cl] = s;
  }
  __syncthreads();
  if (ng == 0 && cl < cw) {
    const float s = (sd[0][cl] + sd[1][cl]) + (sd[2][cl] + sd[3][cl]);
    sd[0][cl] = s * keep_factor(mode, mask, seed, thr, (size_t)p * C + c0 + cl, scale) / (float)HW;
  }
  __syncthreads();
  const int q4 = cw >> 2;
#pragma unroll 4
  for (int i = tid; i < HW * q4; i += HEAD_DG_CH * HEAD_DG_NG) {
    const int hw = i / q4, c = (i - hw * q4) * 4;
    const size_t o = ((size_t)p * HW + hw) * ctot + coff + c0 + c;
    float4 v = *reinterpret_cast<const float4*>(&sd[0][c]);
    if (accumulate) {
      const float4 d = *reinterpret_cast<const float4*>(dx + o);
      v.x += d.x; v.y += d.y; v.z += d.z; v.w += d.w;
    }
    if (act) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(act + o));
      v.x = a.x > 0.f ? v.x : 0.f; v.y = a.y > 0.f ? v.y : 0.f; v.z = a.z > 0.f ? v.z : 0.f; v.w = a.w > 0.f ? v.w : 0.f;
    }
    *reinterpret_cast<float4*>(dx + o) = v;
  }
}

__global__ void segment_mean_fwd_kernel(const float* __restrict__ x, int B, int T, int C, float* __restrict__ out) {
  pdl_sync();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * C) return;
  const int b = i / C, c = i - b * C;
  float s = 0.f;
  for (int t = 0; t < T; ++t) s += __ldg(x + ((size_t)b * T + t) * C + c);
  out[i] = s / (float)T;
}
__global__ void segment_mean_bwd_kernel(const float* __restrict__ dout, int B, int T, int C, float* __restrict__ dx) {
  pdl_sync();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * T * C) return;
  const int c = i % C, b = i / (T * C);
  dx[i] = __ldg(dout + (size_t)b * C + c) / (float)T;
}
__global__ void relu_gate_kernel(const float* __restrict__ grad, const float* __restrict__ act, long long n,
                                 float* __restrict__ out) {
  pdl_sync();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __ldg(act + i) > 0.f ? __ldg(grad + i) : 0.f;
}
// dst[p, dcoff+c, :] = act[p, acoff+c, :] > 0 ? src[p, scoff+c, :] : 0   (ReLU' between channel slices)
__global__ void gate_copy_kernel(const float* __restrict__ src, int sctot, int scoff, const float* __restrict__ act,
                                 int actot, int acoff, float* __restrict__ dst, int dctot, int dcoff, int P, int C,
                                 int HW) {
  pdl_sync();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t total = (size_t)P * C * HW;
  if (i >= total) return;
  const int c = (int)(i % C);
  const size_t ph = i / C;
  const float a = __ldg(act + ph * actot + acoff + c);
  const float v = __ldg(src + ph * sctot + scoff + c);
  dst[ph * dctot + dcoff + c] = a > 0.f ? v : 0.f;
}
// dst[p, coff+c, :] = (relu ? max(.,0) : .)(a[p,c,:] + b[p,c,:])
__global__ void add_relu_slice_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ dst,
                                      int ctot, int coff, int P, int C, int HW, int relu) {
  pdl_sync();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t total = (size_t)P * C * HW;
  if (i >= total) return;
  const int c = (int)(i % C);
  const size_t ph = i / C;
  float v = __ldg(a + i) + __ldg(b + i);
  if (relu) v = fmaxf(v, 0.f);
  dst[ph * ctot + coff + c] = v;
}
__global__ void bias_act_kernel(float* __restrict__ y, const float* __restrict__ bias, int P, int C, int HW, int ctot,
                                int coff, int relu_cols) {
  pdl_sync();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t total = (size_t)P * C * HW;
  if (i >= total) return;
  const int c = (int)(i % C);
  const size_t o = (i / C) * ctot + coff + c;
  float v = y[o] + (bias ? __ldg(bias + c) : 0.f);
  if (c < relu_cols) v = fmaxf(v, 0.f);
  y[o] = v;
}

// weight layouts: canonical OIHW [cout, cin, R, Q] (the reference's state_dict) <-> OHWI [cout, R, Q, cin] (k order of
// the channels-last implicit GEMM).  to_ohwi != 0: dst(OHWI) = src(OIHW); else dst(OIHW) = src(OHWI).
// One block = one output channel x 32 input channels x all taps, staged through shared memory so that both the OIHW
// side (32*rq contiguous floats) and the OHWI side (32 contiguous channels per tap) are accessed coalesced.
__device__ __forceinline__ void permute_weight_block(const float* __restrict__ src, float* __restrict__ dst, int cin, int rq,
                                                     int to_ohwi, int o, int c0, float* tile) {
  const int n = min(32, cin - c0), cnt = n * rq;
  const size_t oihw = ((size_t)o * cin + c0) * rq;      // start of the contiguous OIHW chunk
  const size_t ohwi = (size_t)o * rq * cin + c0;        // element (tap t, channel ci) at ohwi + t*cin + ci
  if (to_ohwi == 1) {
    for (int i = threadIdx.x; i < cnt; i += blockDim.x) tile[i] = __ldg(src + oihw + i);
    __syncthreads();
    for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
      const int t = i / n, ci = i - t * n;
      dst[ohwi + (size_t)t * cin + ci] = tile[ci * rq + t];
    }
  } else {
    for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
      const int t = i / n, ci = i - t * n;
      tile[ci * rq + t] = __ldg(src + ohwi + (size_t)t * cin + ci);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
      if (to_ohwi == 0) dst[oihw + i] = tile[i];
      else dst[oihw + i] += tile[i];                    // 2: accumulate into the OIHW gradient
    }
  }
}
// several weights in one launch: block -> (weight, output channel, 32-channel group)
constexpr int PW_MAX = 16;
struct PermuteBatch {
  int n;
  const float* src[PW_MAX];
  float* dst[PW_MAX];
  int cin[PW_MAX], rq[PW_MAX], cgroups[PW_MAX], blk0[PW_MAX + 1];
};
__global__ void __launch_bounds__(256) permute_weight_batch_kernel(const __grid_constant__ PermuteBatch pb, int to_ohwi) {
  pdl_sync();
  extern __shared__ float tile[];
  int w = 0;
#pragma unroll 1
  while (w + 1 < pb.n && (int)blockIdx.x >= pb.blk0[w + 1]) ++w;
  const int rel = (int)blockIdx.x - pb.blk0[w];
  const int o = rel / pb.cgroups[w], cg = rel - o * pb.cgroups[w];
  permute_weight_block(pb.src[w], pb.dst[w], pb.cin[w], pb.rq[w], to_ohwi, o, cg * 32, tile);
}

static inline unsigned blocks_for(size_t n, int t) { return (unsigned)((n + t - 1) / t); }

}  // namespace offk

using namespace offk;

extern "C" int offk_seed_set(uint64_t* state, uint64_t value, void* stream) {
  OFFK_REQUIRE(state != nullptr, "seed_set: null state");
  (void)launch_pdl(seed_update_kernel, dim3(1), dim3(1), 0, as_stream(stream), state, value);
  return OFFK_LAUNCH_CHECK("seed_set");
}

extern "C" int offk_avgpool_drop_fwd(const float* x, int P, int C, int HW, int x_ctot, int x_coff, int drop_mode,
                                     const uint8_t* keep_mask, uint64_t seed, const uint64_t* seed_dev, float drop_p,
                                     float keep_scale, float* out, void* stream) {
  OFFK_REQUIRE(x && out && P > 0 && C > 0 && HW > 0 && x_coff >= 0 && x_coff + C <= x_ctot, "avgpool_fwd: bad args");
  OFFK_REQUIRE(drop_mode != OFFK_DROP_MASK || keep_mask, "avgpool_fwd: mask missing");
  (void)launch_pdl(avgpool_drop_fwd_kernel, dim3(blocks_for((size_t)P * C, 128)), dim3(128), 0, as_stream(stream), 
      x, P, C, HW, x_ctot, x_coff, drop_mode, keep_mask, seed, seed_dev, drop_p, keep_scale, out);
  return OFFK_LAUNCH_CHECK("avgpool_drop_fwd");
}

extern "C" int offk_pool3_nhwc(const float* x, int n_img, int H, int W, int x_ctot, int x_coff, int C, int stride, int pad,
                               int kind, float* y, int y_ctot, int y_coff, void* stream) {
  OFFK_REQUIRE(x && y && n_img > 0 && H > 0 && W > 0 && C > 0 && stride >= 1 && pad >= 0 && 2 * pad < 3 &&
                   (kind == OFFK_POOL_MAX || kind == OFFK_POOL_AVG),
               "pool3_nhwc: bad args");
  OFFK_REQUIRE(C % 4 == 0 && x_ctot % 4 == 0 && x_coff % 4 == 0 && y_ctot % 4 == 0 && y_coff % 4 == 0 && x_coff + C <= x_ctot &&
                   y_coff + C <= y_ctot && ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15u) == 0,
               "pool3_nhwc: channel slices must be 16-byte aligned quads");
  // ceil mode: ceil((H + 2 pad - 3) / stride) + 1 windows, the last of which must start inside the input or its left padding
  int Ho = (H + 2 * pad - 3 + stride - 1) / stride + 1, Wo = (W + 2 * pad - 3 + stride - 1) / stride + 1;
  if ((Ho - 1) * stride >= H + pad) --Ho;
  if ((Wo - 1) * stride >= W + pad) --Wo;
  OFFK_REQUIRE(Ho >= 1 && Wo >= 1, "pool3_nhwc: input smaller than the window");
  // count_include_pad divides by 9 only while every window stays inside the padded input
  OFFK_REQUIRE(kind == OFFK_POOL_MAX || ((Ho - 1) * stride + 3 <= H + 2 * pad && (Wo - 1) * stride + 3 <= W + 2 * pad),
               "pool3_nhwc: an average window runs past the padded input");
  const long long total = (long long)n_img * Ho * Wo * (C / 4);
  (void)launch_pdl(pool3_nhwc_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, as_stream(stream), x, H, W, x_ctot,
                   x_coff, C / 4, stride, pad, kind, Ho, Wo, total, y, y_ctot, y_coff);
  return OFFK_LAUNCH_CHECK("pool3_nhwc");
}

extern "C" int offk_image_to_nhwc(const float* src, float* dst, int n_img, int c, int hw, int c_pad, void* stream) {
  OFFK_REQUIRE(src && dst && n_img > 0 && hw > 0 && c > 0 && c <= c_pad && c_pad % 4 == 0 &&
                   (reinterpret_cast<uintptr_t>(dst) & 15u) == 0,
               "image_to_nhwc: bad args (0 < c <= c_pad, c_pad %% 4 == 0, 16-byte aligned dst)");
  const long long total = (long long)n_img * hw;
  (void)launch_pdl(image_to_nhwc_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, as_stream(stream), src, dst, c, hw,
                   c_pad, total);
  return OFFK_LAUNCH_CHECK("image_to_nhwc");
}

extern "C" int offk_head_fwd(const float* x, int P, int C, int HW, int x_ctot, int x_coff, int drop_mode, const uint8_t* keep_mask,
                             uint64_t seed, const uint64_t* seed_dev, float drop_p, float keep_scale, const float* weight,
                             const float* bias, int num_classes, int T, float* pooled, float* out, float* consensus_out,
                             void* stream) {
  OFFK_REQUIRE(x && weight && bias && out && P > 0 && HW > 0 && num_classes > 0 && num_classes <= 128, "head_fwd: bad args");
  OFFK_REQUIRE(C > 0 && C <= HEAD_MAX_C && C % 4 == 0 && x_coff >= 0 && x_coff % 4 == 0 && x_ctot % 4 == 0 && x_coff + C <= x_ctot &&
                   (reinterpret_cast<uintptr_t>(x) & 15u) == 0,
               "head_fwd: channel slice (C, x_coff, x_ctot multiples of 4, C <= 1024, 16-byte aligned x)");
  OFFK_REQUIRE(T >= 1 && P % T == 0 && (T == 1 || consensus_out), "head_fwd: T must divide P; T > 1 needs consensus_out");
  OFFK_REQUIRE(drop_mode != OFFK_DROP_MASK || keep_mask, "head_fwd: mask missing");
  OFFK_REQUIRE((reinterpret_cast<uintptr_t>(weight) & 15u) == 0, "head_fwd: weight alignment");
  (void)launch_pdl(head_fwd_kernel, dim3(P / T), dim3(HEAD_THREADS), 0, as_stream(stream), x, C, HW, x_ctot, x_coff, drop_mode,
                   keep_mask, seed, seed_dev, drop_p, keep_scale, weight, bias, num_classes, T, pooled, out, consensus_out);
  return OFFK_LAUNCH_CHECK("head_fwd");
}

extern "C" int offk_head_bwd(const float* dout, int P, int C, int HW, int ctot, int coff, int drop_mode, const uint8_t* keep_mask,
                             uint64_t seed, const uint64_t* seed_dev, float drop_p, float keep_scale, const float* weight,
                             int num_classes, int T, const float* pooled, const float* act, int accumulate, float* dx,
                             float* dweight, float* dbias, void* stream) {
  OFFK_REQUIRE(dout && weight && P > 0 && HW > 0 && num_classes > 0 && num_classes <= 128, "head_bwd: bad args");
  OFFK_REQUIRE(C > 0 && C <= HEAD_MAX_C && C % 4 == 0 && coff >= 0 && coff % 4 == 0 && ctot % 4 == 0 && coff + C <= ctot,
               "head_bwd: channel slice (multiples of 4, C <= 1024)");
  OFFK_REQUIRE(T >= 1 && P % T == 0, "head_bwd: T must divide P");
  OFFK_REQUIRE(drop_mode != OFFK_DROP_MASK || keep_mask, "head_bwd: mask missing");
  if (dweight) {
    OFFK_REQUIRE(pooled != nullptr, "head_bwd: the weight gradient needs the pooled features of the forward pass");
    (void)launch_pdl(head_wgrad_kernel, dim3((C + 127) / 128, (num_classes + 7) / 8, (P + HEAD_WG_PAIRS - 1) / HEAD_WG_PAIRS), dim3(128, 8), 0, as_stream(stream), dout, pooled,
                     P, C, num_classes, T, dweight, dbias);
    if (int e = OFFK_LAUNCH_CHECK("head_wgrad")) return e;
  }
  if (dx) {
    OFFK_REQUIRE((reinterpret_cast<uintptr_t>(dx) & 15u) == 0, "head_bwd: dx alignment");
    (void)launch_pdl(head_dgrad_kernel, dim3(P, (C + HEAD_DG_CH - 1) / HEAD_DG_CH), dim3(HEAD_DG_CH * HEAD_DG_NG), 0, as_stream(stream), dout, weight, C, HW, ctot, coff,
                     num_classes, T, drop_mode, keep_mask, seed, seed_dev, drop_p, keep_scale, act, accumulate, dx);
    if (int e = OFFK_LAUNCH_CHECK("head_dgrad")) return e;
  }
  return 0;
}

extern "C" int offk_segment_mean_fwd(const float* x, int B, int T, int C, float* out, void* stream) {
  OFFK_REQUIRE(x && out && B > 0 && T > 0 && C > 0, "segment_mean_fwd: bad args");
  (void)launch_pdl(segment_mean_fwd_kernel, dim3(blocks_for((size_t)B * C, 256)), dim3(256), 0, as_stream(stream), x, B, T, C, out);
  return OFFK_LAUNCH_CHECK("segment_mean_fwd");
}
extern "C" int offk_segment_mean_bwd(const float* dout, int B, int T, int C, float* dx, void* stream) {
  OFFK_REQUIRE(dout && dx && B > 0 && T > 0 && C > 0, "segment_mean_bwd: bad args");
  (void)launch_pdl(segment_mean_bwd_kernel, dim3(blocks_for((size_t)B * T * C, 256)), dim3(256), 0, as_stream(stream), dout, B, T, C, dx);
  return OFFK_LAUNCH_CHECK("segment_mean_bwd");
}
extern "C" int offk_relu_gate(const float* grad, const float* act, long long n, float* out, void* stream) {
  OFFK_REQUIRE(grad && act && out && n > 0, "relu_gate: bad args");
  (void)launch_pdl(relu_gate_kernel, dim3(blocks_for((size_t)n, 256)), dim3(256), 0, as_stream(stream), grad, act, n, out);
  return OFFK_LAUNCH_CHECK("relu_gate");
}
extern "C" int offk_bias_act(float* y, const float* bias, int P, int C, int HW, int ctot, int coff, int relu_cols,
                             void* stream) {
  OFFK_REQUIRE(y && P > 0 && C > 0 && HW > 0 && coff >= 0 && coff + C <= ctot, "bias_act: bad args");
  (void)launch_pdl(bias_act_kernel, dim3(blocks_for((size_t)P * C * HW, 256)), dim3(256), 0, as_stream(stream), y, bias, P, C, HW, ctot, coff,
                                                                                     relu_cols);
  return OFFK_LAUNCH_CHECK("bias_act");
}

extern "C" int offk_gate_copy(const float* src, int src_ctot, int src_coff, const float* act, int act_ctot,
                              int act_coff, float* dst, int dst_ctot, int dst_coff, int P, int C, int HW,
                              void* stream) {
  OFFK_REQUIRE(src && act && dst && P > 0 && C > 0 && HW > 0, "gate_copy: bad args");
  OFFK_REQUIRE(src_coff + C <= src_ctot && act_coff + C <= act_ctot && dst_coff + C <= dst_ctot, "gate_copy: slices");
  (void)launch_pdl(gate_copy_kernel, dim3(blocks_for((size_t)P * C * HW, 256)), dim3(256), 0, as_stream(stream), 
      src, src_ctot, src_coff, act, act_ctot, act_coff, dst, dst_ctot, dst_coff, P, C, HW);
  return OFFK_LAUNCH_CHECK("gate_copy");
}

extern "C" int offk_add_relu_slice(const float* a, const float* b, float* dst, int dst_ctot, int dst_coff, int P,
                                   int C, int HW, int relu, void* stream) {
  OFFK_REQUIRE(a && b && dst && P > 0 && C > 0 && HW > 0 && dst_coff >= 0 && dst_coff + C <= dst_ctot,
               "add_relu_slice: bad args");
  (void)launch_pdl(add_relu_slice_kernel, dim3(blocks_for((size_t)P * C * HW, 256)), dim3(256), 0, as_stream(stream), a, b, dst, dst_ctot,
                                                                                           dst_coff, P, C, HW, relu);
  return OFFK_LAUNCH_CHECK("add_relu_slice");
}

extern "C" int offk_fill_zero(float* p, long long n, void* stream) {
  OFFK_REQUIRE(p != nullptr && n >= 0, "fill_zero: bad args");
  if (n == 0) return 0;
  return cuda_check(cudaMemsetAsync(p, 0, (size_t)n * sizeof(float), as_stream(stream)), "fill_zero");
}

// dst[i] = src[idx[i]]: all per-step weight re-layouts (OHWI forward copies, flipped / transposed data-gradient copies)
// in one launch; idx is built once per plan on the host
__global__ void gather_copy_kernel(const float* __restrict__ src, const int32_t* __restrict__ idx, float* __restrict__ dst,
                                   long long n) {
  pdl_sync();
  const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i + 3 < n) {
    const int4 j = *reinterpret_cast<const int4*>(idx + i);
    *reinterpret_cast<float4*>(dst + i) = make_float4(__ldg(src + j.x), __ldg(src + j.y), __ldg(src + j.z), __ldg(src + j.w));
  } else {
    for (long long k = i; k < n; ++k) dst[k] = __ldg(src + idx[k]);
  }
}

// NCHW [n, C, HW] -> channels-last [n, HW, C] through 32x32 shared-memory tiles (both sides coalesced)
__global__ void __launch_bounds__(256) nchw_to_nhwc_kernel(const float* __restrict__ src, float* __restrict__ dst, int C, int HW) {
  pdl_sync();
  __shared__ float t[32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const size_t img = blockIdx.z;
  const float* s = src + img * (size_t)C * HW;
  float* d = dst + img * (size_t)C * HW;
#pragma unroll
  for (int j = ty; j < 32; j += 8) {
    const int c = c0 + j, p = p0 + tx;
    if (c < C && p < HW) t[j][tx] = __ldg(s + (size_t)c * HW + p);
  }
  __syncthreads();
#pragma unroll
  for (int j = ty; j < 32; j += 8) {
    const int p = p0 + j, c = c0 + tx;
    if (p < HW && c < C) d[(size_t)p * C + c] = t[tx][j];
  }
}

extern "C" int offk_nchw_to_nhwc(const float* src, float* dst, int n_img, int C, int HW, void* stream) {
  OFFK_REQUIRE(src && dst && n_img > 0 && C > 0 && HW > 0 && n_img <= 65535, "nchw_to_nhwc: bad args");
  dim3 grid((HW + 31) / 32, (C + 31) / 32, n_img);
  OFFK_REQUIRE(grid.y <= 65535, "nchw_to_nhwc: too many channels");
  (void)launch_pdl(nchw_to_nhwc_kernel, dim3(grid), dim3(256), 0, as_stream(stream), src, dst, C, HW);
  return OFFK_LAUNCH_CHECK("nchw_to_nhwc");
}

extern "C" int offk_gather_copy(const float* src, const int32_t* idx, float* dst, long long n, void* stream) {
  OFFK_REQUIRE(src && idx && dst && n >= 0, "gather_copy: bad args");
  OFFK_REQUIRE((reinterpret_cast<uintptr_t>(idx) & 15u) == 0 && (reinterpret_cast<uintptr_t>(dst) & 15u) == 0, "gather_copy: alignment");
  if (n == 0) return 0;
  const long long threads = (n + 3) / 4;
  (void)launch_pdl(gather_copy_kernel, dim3((unsigned)((threads + 255) / 256)), dim3(256), 0, as_stream(stream), src, idx, dst, n);
  return OFFK_LAUNCH_CHECK("gather_copy");
}

extern "C" int offk_permute_weight_batch(int n, const offk_permute_t* items, int to_ohwi, void* stream) {
  OFFK_REQUIRE(n >= 1 && n <= PW_MAX && items != nullptr, "permute_weight_batch: 1 <= n <= %d", PW_MAX);
  PermuteBatch pb;
  pb.n = n;
  long long blk = 0;
  int rq_max = 0;
  for (int i = 0; i < n; ++i) {
    const offk_permute_t& it = items[i];
    OFFK_REQUIRE(it.src && it.dst && it.cout > 0 && it.cin > 0 && it.kh > 0 && it.kw > 0 && it.kh * it.kw <= 256, "permute_weight_batch: item %d", i);
    pb.src[i] = it.src; pb.dst[i] = it.dst; pb.cin[i] = it.cin; pb.rq[i] = it.kh * it.kw;
    pb.cgroups[i] = (it.cin + 31) / 32;
    pb.blk0[i] = (int)blk;
    blk += (long long)pb.cgroups[i] * it.cout;
    if (pb.rq[i] > rq_max) rq_max = pb.rq[i];
  }
  pb.blk0[n] = (int)blk;
  OFFK_REQUIRE(blk < 2147483647LL, "permute_weight_batch: grid too large");
  (void)launch_pdl(permute_weight_batch_kernel, dim3((unsigned)blk), dim3(256), (size_t)32 * rq_max * sizeof(float), as_stream(stream), pb, to_ohwi);
  return OFFK_LAUNCH_CHECK("permute_weight_batch");
}
