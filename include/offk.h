/*
 * offk.h -- C ABI of liboffk.so, the sm_100a kernels behind the OFF
 * (Optical Flow guided Feature) unit and OFF sub-network.
 *
 * The reference (JoeHEZHAO/Optical-Flow-Guided-Feature-Pytorch) has no FFI
 * layer of its own: its boundary is the nn.Module surface and every op on the
 * path is a stock ATen call (SURVEY.md section 2b).  Each entry point below
 * therefore names the reference call sites it replaces (file:line into the
 * reference repository).  INTEGRATION.md shows the ctypes binding a maintainer
 * of the reference would add.
 *
 * Conventions
 *   - plain C: raw device pointers, ints, an opaque stream (cudaStream_t cast
 *     to void*).  No torch types.  All tensors fp32, NCHW, caller-owned.
 *   - the library never allocates or frees device memory and never keeps a
 *     pointer past the call; every call is asynchronous on `stream` and safe
 *     under CUDA-graph capture.
 *   - return 0 on success; a positive cudaError_t or a negative OFFK_E_* code
 *     otherwise.  offk_last_error_string() describes the last failure of the
 *     calling thread.  No exceptions, no exit().
 */
#ifndef OFFK_H_
#define OFFK_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OFFK_VERSION 100 /* 0.1.0 */

#define OFFK_E_BADARG   (-1)  /* shape / alignment / null-pointer violation */
#define OFFK_E_NOTSM100 (-2)  /* device is not compute capability 10.x       */
#define OFFK_E_LIMIT    (-3)  /* size beyond what the kernel supports        */

/* arithmetic of the dense contractions */
#define OFFK_PREC_TF32   1 /* tcgen05.mma kind::tf32, operands in smem, fp32 accumulate in TMEM                        */
#define OFFK_PREC_TF32X3 2 /* fp32-parity mode on the tensor cores (the reference computes in fp32, RGB_OFF.py:597):
                              every operand tile x is used as hi = trunc_tf32(x) (what kind::tf32 reads anyway) plus a
                              residual tile lo = tf32(x - hi) produced in shared memory, and three MMAs
                              A_lo*B_hi + A_hi*B_lo + A_hi*B_hi accumulate into the same fp32 TMEM tile ("3xTF32") */

/* which frame feeds the spatial branch of pair p=(b,t) (SURVEY.md 3.3) */
#define OFFK_INDEX_REFERENCE_FLAT 0 /* flat frame p, as RGB_OFF.py:609 literally does */
#define OFFK_INDEX_ALIGNED        1 /* frame (b,t)                                    */

/* dropout on the spatial-gradient channels / pooled head features */
#define OFFK_DROP_NONE 0
#define OFFK_DROP_MASK 1 /* caller-supplied uint8 keep-mask (1 = keep)             */
#define OFFK_DROP_SEED 2 /* counter-hash keep decision from (seed, element index)   */
/* OFFK_DROP_SEED element index: channels-last, ((p*H*W + pix) * K*Cs + channel) for the spatial-gradient channels
 * of pair p, p*C + c for pooled head features; four consecutive indices share one 64-bit hash
 * (offk_drop_keep_host mirrors the device decision). */

int offk_version(void);
const char* offk_last_error_string(void);
/* fills sm_count, cc_major, cc_minor, l2_bytes of the current device */
int offk_device_info(int* sm_count, int* cc_major, int* cc_minor, long long* l2_bytes);

/* ------------------------------------------------------------------------
 * Gather-GEMM:  D[m,n] = sum_k A(m,k) * B(n,k),  then a fused epilogue.
 *
 * The contractions whose operands no TMA tensor map describes (offk_tma_gemm below carries every forward conv and
 * every stage-conv data gradient).  The engine launches it for
 *   - the weight gradients of the stage convs (RGB_OFF.py:657-685,762-780,833-841; autograd, train_off.py:136-146) in
 *     the tf32 mode, except motion_conv_trans_28: A = im2col(x)^T and B = dY, both OFFK_LOAD_VEC_ROW, out_vec = 2
 *     (dW rows contiguous) and the all-ones row for the bias gradient, with or without split-K;
 *   - the data gradients of the nine OFF units' fused 1x1 conv (RGB_OFF.py:597,610 ...) into the NCHW taps, when the
 *     caller asks for tap gradients: A = dY (OFFK_LOAD_VEC_K), B = the weights (OFFK_LOAD_VEC_ROW), a plain store
 *     through the out tables.
 * The other two pairings of the load modes are accepted as well; tables.py picks a mode from each operand's layout.
 * What differs per layer is only WHERE element (m,k) / (n,k) / (m,n) lives;
 * that is described by separable index tables built once per layer geometry
 * (by the host: optical-flow-guided-feature-pytorch_b200/tables.py builds them with numpy for forward,
 * weight-gradient and data-gradient of a conv in NCHW or channels-last layout):
 *
 *   A(m,k) = a_src[a_row[m].off + a_col[k].off]   if 0 <= a_row[m].y + a_col[k].y < a_h
 *                                                 and 0 <= a_row[m].x + a_col[k].x < a_w, else 0
 *            (a_h == 0 disables the box test; a_ones_row == m gives A(m,.) = 1 -> bias gradient)
 *   B(n,k) = b_src[b_row[n] + b_col[k]]
 *   out[out_row[m] + out_col[n]]  receives the epilogue of D[m,n].
 *
 * Epilogue, in this order, each step optional:
 *   v = D[m,n] + bias[n]
 *   v = max(v,0)                         if n <  relu_pre_cols
 *   v = gate[o] > 0 ? v : 0              if gate && gate_first  && n >= gate_col0   (ReLU')
 *   v = v + addend[add_row[m] + add_col[n]]   if addend
 *   v = gate[o] > 0 ? v : 0              if gate && !gate_first && n >= gate_col0
 *   v = max(v,0)                         if relu_post
 *   out[o] = v   (atomic add when split_k > 1 or atomic_out; then bias / activations are NOT applied)
 * o = out_row[m] + out_col[n]: the gate is read at the output's own element.  A NULL add_row / add_col stands for the
 * out table.
 *
 * Table padding contract (so the kernels never bounds-check an index): a_row has ceil(M/128)*128 entries, a_col
 * and b_col have ceil(K/32)*32 + 64 entries, b_row has ceil(N/256)*256 entries.  Padding entries of a_row /
 * a_col carry y = -16384 (the box test is always on; pass a_h = a_w = 32767 for "no box"), padding entries of
 * b_row / b_col are 0.  The entry of a_ones_row is never gathered.
 * ---------------------------------------------------------------------- */
/* Operand fetch modes.  The tables are always element-granular; a load mode is a promise by the caller
 * that groups of 4 consecutive indices are contiguous in memory, 16-byte aligned and share validity
 * (a_src and b_src 16-byte aligned).  An operand without such groups cannot be launched. */
#define OFFK_LOAD_VEC_K      2 /* 16-byte loads of 4 consecutive k (K % 4 == 0): NHWC activations, dense weights */
#define OFFK_LOAD_VEC_ROW    3 /* 16-byte cp.async of 4 consecutive rows straight into the MN-major swizzled tile (the
                                  operand is then marked MN-major for tcgen05.mma; nothing is transposed): NCHW taps
                                  as A(m = pixel), channels-last tensors in weight- and data-gradient GEMMs        */

typedef struct offk_idx {
  int32_t off; /* element offset contribution                        */
  int16_t y;   /* row coordinate contribution for the validity box   */
  int16_t x;   /* column coordinate contribution                     */
} offk_idx_t;

typedef struct offk_gemm {
  int32_t M, N, K;
  /* A operand */
  const float* a_src;
  const offk_idx_t* a_row; /* [M] */
  const offk_idx_t* a_col; /* [K] */
  int32_t a_h, a_w;        /* validity box (>= 1); 32767 = every real element is valid */
  int32_t a_ones_row;      /* -1, or the row whose A values are all 1 */
  int32_t a_mode;          /* OFFK_LOAD_*: how the producer warps may fetch this operand */
  /* B operand */
  const float* b_src;
  const int32_t* b_row; /* [N] */
  const int32_t* b_col; /* [K] */
  int32_t b_mode;       /* OFFK_LOAD_* */
  /* epilogue */
  float* out;
  const int32_t* out_row; /* [M] */
  const int32_t* out_col; /* [N] */
  const float* bias;      /* [N] or NULL */
  int32_t relu_pre_cols;
  const float* gate;
  int32_t gate_col0;
  int32_t gate_first;
  const float* addend;
  const int32_t* add_row;
  const int32_t* add_col;
  int32_t relu_post;
  int32_t atomic_out;
  float* ones_row_out; /* wgrad: D[a_ones_row, n] accumulates into ones_row_out[n] (bias gradient) */
  int32_t split_k;     /* >= 1; > 1 forces atomic accumulation into a zero-initialised `out` */
  int32_t tile_n;      /* 0 = auto; else the N tile of the tensor-core kernel (multiple of 16, <= 256) */
  int32_t out_vec;     /* 1: out/gate/addend are contiguous along n (out_col[n] = out_col[0] + n, N % 4 == 0, all
                          offsets and bias 16-byte aligned): float4 epilogue (NHWC outputs)
                          2: out is contiguous along m (out_row[m] = out_row[0] + m with out_row[0] % 4 == 0, every
                          out_col[n] % 4 == 0, `out` 16-byte aligned; no bias / gate / addend): the tensor-core kernels
                          transpose the tile and add 4 consecutive rows per lane (weight gradients: dW[n][m]) */
  int32_t reserved;
  /* offk_tma_gemm with out_vec = 1 only (NULL / 0 elsewhere):
   * finish_counter: split-K without a second kernel.  One int per output tile (tile = blockIdx.y * gridDim.x + blockIdx.x;
   *   zero before the first launch, left zero by every launch).  The split CTAs add their partial tiles into the
   *   zero-initialised `out`; the last one to arrive re-reads the summed tile and applies the epilogue above (bias, ReLU
   *   prefix, gate, addend, ReLU) in place -- so bias / activation ARE applied although split_k > 1.
   * aux_out: a second output written where the final value v of an element is produced (directly, or by the split-K
   *   finisher):  aux_out[aux_row[m] + n] = max(v + aux_addend[out_row[m] + out_col[n]], 0)
   *   (aux_row NULL: the out_row table; aux_addend NULL: 0).  RGB_OFF.py:658 (the ReLU'd copy of motion_conv_trans_28's
   *   pre-activation output, which :665 also consumes raw) and :779-780,832 (sum_14b = relu(sum_14a + relu(conv3_14b)) written
   *   into the 7x7 fusion buffer while the inner ReLU output is kept for the backward pass). */
  int32_t* finish_counter;
  float* aux_out;
  const int32_t* aux_row;
  const float* aux_addend;
} offk_gemm_t;

int offk_gather_gemm(const offk_gemm_t* g, int precision, void* stream);

/* ------------------------------------------------------------------------
 * TMA-fed GEMM: the same contraction and epilogue as offk_gather_gemm (bias, ReLU prefix, ReLU' gate, residual
 * add, split-K / atomic accumulation, output through out_row / out_col), but the operand tiles are fetched by the
 * Tensor Memory Accelerator (cp.async.bulk.tensor) instead of index-table gathers.  Used for the fused 1x1 conv of the
 * nine OFF units on the NCHW taps (RGB_OFF.py:597-598,609-610 and the eight copies) and its weight gradient, for every
 * conv / FC of the OFF sub-network whose input is a channels-last activation -- the residual-block 1x1 convs and FC
 * heads (:659-685,764-780,787,793,835-847) as dense 2-D tiles, the stage-entry 7x7/5x5/3x3 convs and the bottleneck
 * 3x3s (:657,661,672,681,762,766,775,777,833,837) through TMA im2col mode -- and for their data gradients (autograd,
 * train_off.py:136-146): a stride-1 conv's dX is a conv over dY with flipped weights, a stride-2 conv's dX is one
 * OFFK_TGEMM_FREE_GEOM correlation over dY per stride-parity class of the input pixel.
 *   g.a_src / g.b_src : operand base pointers (16-byte aligned); the a_row/a_col/b_row/b_col tables are ignored
 *   A dense  : A(m,k) = a_src[m*lda + k]
 *   A im2col : a_src = channels-last [n_img, hin, win, ctot]; channels [a_coff, a_coff+cin) feed the conv;
 *              K = kh*kw*cin ordered (r, q, c) -- the order of OHWI weights; cin % 32 == 0
 *   A nchw   : a_src = NCHW [n_img, cin, hin*win] (pixels contiguous); fetched as the MN-major tcgen05 operand, so the
 *              NCHW -> channels-last conversion of the unit's fused 1x1 conv executes no transpose
 *   B dense  : B(n,k) = b_src[n*ldb + k]   (weights [cout, K])
 *   weight-gradient kinds (A nchw_t / im2col_t with B dense_t): see the OFFK_TMA_* definitions below; the all-ones
 *   row g.a_ones_row (bias gradient) is synthesised inside the kernel; out_vec is 0 or 2 (rows contiguous)
 *   with out_vec = 1 the out / gate / addend column tables must be contiguous (col[n] = col[0] + n)
 * offk_tma_gemm_prepare() encodes the two CUtensorMap objects into the descriptor (host only, no device memory);
 * call it again whenever a pointer or shape changes.  t->precision selects OFFK_PREC_TF32 or OFFK_PREC_TF32X3.
 * ---------------------------------------------------------------------- */
#define OFFK_TMA_A_DENSE  0
#define OFFK_TMA_A_IM2COL 1
#define OFFK_TMA_A_NCHW   2 /* A(m = img*hw + pix, k = c) = a_src[(img*cin + c)*hw + pix]: an NCHW tensor read in place
                               (the BN-Inception taps of motion_conv_gen_X / motion_spatial_down_X, RGB_OFF.py:597,610);
                               hw = hin*win, hw % 4 == 0, cin % 32 == 0; M tiles are cut per frame */
#define OFFK_TMA_A_NCHW_T   3 /* weight gradient of the above: A(m = c, k = img*hw + pix), same NCHW tensor; M = cin (+ 1:
                                 a_ones_row == cin gives the bias gradient); K-blocks are cut per frame */
#define OFFK_TMA_A_IM2COL_T 4 /* weight gradient of a channels-last conv: A(m = (r,q,c), k = output pixel) = im2col(x)^T;
                                 M = kh*kw*cin (+ 1: a_ones_row == kh*kw*cin); cin % 32 == 0 */
#define OFFK_TMA_B_DENSE  0
#define OFFK_TMA_B_DENSE_T 1  /* B(n,k) = b_src[k*ldb + n]: a row-major [K, ldb] matrix (the channels-last output gradient
                                 dY[pixel, cout slice] of a weight-gradient GEMM).  Pairs with the *_T A kinds. */

#define OFFK_TGEMM_FREE_GEOM 1

typedef struct offk_tgemm {
  offk_gemm_t g;
  int32_t a_kind, lda, a_coff;
  int32_t n_img, hin, win, ctot, cin, kh, kw, stride, pad, hout, wout; /* im2col geometry */
  int32_t b_kind, ldb;
  int32_t prepared;      /* set by offk_tma_gemm_prepare (the N tile the B tensor map was built for) */
  int32_t geom_flags;    /* OFFK_TGEMM_FREE_GEOM: hout / wout are given (not derived), pad = top rows, pad_w = left columns,
                            kh != kw allowed -- the data gradient of a strided conv, one stride-parity class at a time, is
                            such a stride-1 correlation over dY (autograd of RGB_OFF.py:657,762) */
  int32_t pad_w;
  int32_t precision;     /* OFFK_PREC_TF32 (or 0) / OFFK_PREC_TF32X3 */
  int32_t bk;            /* K-block depth: 0 / 32, or 64 / 128 for OFFK_TMA_A_IM2COL_T (both operands MN-major: deeper K-blocks
                            = fewer, larger TMA boxes; fixed before offk_tma_gemm_prepare) */
  int32_t reserved;
  int64_t b_lo_delta;    /* OFFK_PREC_TF32X3 with OFFK_TMA_B_DENSE: 0, or the element distance from B to a matrix of the same
                            layout holding its tf32 residuals (offk_tf32_residual): the weights are then split once per step in
                            global memory and both tiles arrive by TMA, instead of every CTA splitting the weight tile of every
                            K-block in shared memory; a positive multiple of 4 */
  int32_t out_ld;        /* > 0 (with g.out_vec = 1): the output rows are linear, out_row[m] == m * out_ld, and the columns
                            start at element out_c0 (== out_col[0]).  A plain epilogue (bias / ReLU only, or raw split-K
                            partial sums; no gate, addend, finisher or second output) whose N tile is a multiple of 32
                            then leaves through the TMA: the tile is staged in shared memory in 32-column slabs and
                            written with cp.async.bulk.tensor stores (cp.reduce...add for split-K); st.global from the
                            eight epilogue warps sustains only ~12 B/clock/SM (profiles/timeline_*_r02n.txt).
                            0 = always st.global / red.global. */
  int32_t out_c0;
  uint64_t tmap_a[16];   /* CUtensorMap storage */
  uint64_t tmap_b[16];
  uint64_t tmap_c[16];   /* output map (offk_tma_gemm_prepare; used when c_mode != 0) */
  int32_t c_mode;        /* set by offk_tma_gemm_prepare: 0 = no TMA stores, 1 = 2-D {N, M}, 2 = 3-D {N, hw, n_img} (A nchw) */
  int32_t reserved3;
} offk_tgemm_t;

int offk_tma_gemm_prepare(offk_tgemm_t* t);
int offk_tma_gemm(const offk_tgemm_t* t, void* stream);

/* ------------------------------------------------------------------------
 * Fused OFF stencil: spatial gradient + temporal difference + dropout +
 * both torch.cat()s in one pass.  Replaces RGB_OFF.py:599-604 (view / slice /
 * sub), :611 (depth-wise 3x3, learned weight + bias) or Flow_OFF.py:622
 * (fixed diagonal kernel) or util.py:46-50 (Sobel x and y, K = 2), :612
 * (dropout), :616 (cat) and the stage cats :656,:760,:832.
 *
 * Tensors are channels-last (the library's internal layout; the reference's NCHW taps are converted by the
 * unit's 1x1 GEMM epilogue):
 *   g : reduced+ReLU'd features  G[f, y, x, c]  f in [0,B*L), c in [0,Cg); frame stride g_fs, pixel stride g_ps floats
 *   d : spatial-branch features  D[f, y, x, c]  c in [0,Cs);              frame stride d_fs, pixel stride d_ps
 *   w : [Cs, K, 3, 3] cross-correlation taps, bias [Cs*K] or NULL
 *   out: [P, H, W, out_ctot]
 *   out[p, y, x, out_coff + kk*Cs + c] = drop( sum_ij w[c,kk,i,j] * D[fs(p), y+i-1, x+j-1, c] + bias )   (zero pad)
 *   out[p, y, x, out_coff + K*Cs + c]  = G[b*L+t+1, y, x, c] - G[b*L+t, y, x, c]        p = b*(L-1)+t
 *   keep_mask is indexed like the reference's dropout input [P, K*Cs, H, W] (RGB_OFF.py:612); seeded dropout hashes
 *   the channels-last element index (see OFFK_DROP_SEED)
 *   fs(p) = p (OFFK_INDEX_REFERENCE_FLAT) or b*L+t (OFFK_INDEX_ALIGNED)
 * Each G frame is read once.  Cg == 0 or Cs == 0 disables a half (the
 * stand-alone util.SobelFilter modules use Cg == 0, L == 2 so that p == f).
 * ---------------------------------------------------------------------- */
typedef struct offk_stencil {
  int32_t B, L, Cg, Cs, K, H, W;
  int64_t g_fs, d_fs;      /* frame strides (floats) of g and d */
  int32_t g_ps, d_ps;      /* pixel strides (floats) of g and d: channels-last [f, y, x, c] */
  int32_t out_ctot, out_coff;
  int32_t index_mode;
  int32_t drop_mode;       /* OFFK_DROP_* */
  float keep_scale;        /* 1/(1-p) */
  float drop_p;            /* p, used by OFFK_DROP_SEED */
  uint64_t seed;
  const uint8_t* keep_mask; /* [P, K*Cs, H, W] (NCHW order) for OFFK_DROP_MASK */
  const uint64_t* seed_dev; /* OFFK_DROP_SEED: NULL, or a device word added to `seed` when the kernel runs -- the per-step
                               part of the seed then lives in device memory (offk_seed_set), so a captured CUDA graph
                               draws fresh masks on every replay while `seed` stays the call site's salt */
} offk_stencil_t;

int offk_stencil_diff_fwd(const offk_stencil_t* s, const float* g, const float* d, const float* w,
                          const float* bias, float* out, void* stream);

/* Buffers of one OFF unit for the batched entry points below (forward uses g, d, w, bias, out; backward uses
 * dout, g, d, w, dg, dg_fs, dd, dd_fs, dw, dbias -- same meaning as the single-unit calls). */
typedef struct offk_stencil_io {
  const float* g;
  const float* d;
  const float* w;
  const float* bias;
  float* out;
  const float* dout;
  float* dg;
  int64_t dg_fs;
  float* dd;
  int64_t dd_fs;
  float* dw;
  float* dbias;
} offk_stencil_io_t;

/* n (<= 12) OFF units in ONE launch: the units that feed one stage-fusion buffer (RGB_OFF.py:656: 3a,3b; :760:
 * 3c,4a,4b,4c,4d; :832: 5a,5b), so the small 14x14 / 7x7 levels do not pay a launch latency each.  s and io are
 * host arrays of n entries; semantics per entry are those of offk_stencil_diff_fwd / _bwd. */
int offk_stencil_diff_fwd_batch(int n, const offk_stencil_t* s, const offk_stencil_io_t* io, void* stream);
int offk_stencil_diff_bwd_batch(int n, const offk_stencil_t* s, const offk_stencil_io_t* io, void* stream);

/* Backward of the above.  dout is the gradient of the stage buffer (same
 * ctot/coff addressing as `out`).  Writes
 *   dg[f,c,:,:] = (dT[b,t-1] - dT[b,t]) * (G[f,c,:,:] > 0)      (ReLU' of RGB_OFF.py:598 folded in)
 *   dd[f,c,:,:] = transpose-stencil of the dropped spatial gradient (0 for frames that feed no pair)
 * and accumulates (atomicAdd into zero-initialised buffers) dw [Cs,K,3,3], dbias [Cs*K] when non-NULL.
 * g is read for the ReLU mask, d for the weight gradient.  dg/dd frame strides: dg_fs, dd_fs. */
int offk_stencil_diff_bwd(const offk_stencil_t* s, const float* dout, const float* g, const float* d,
                          const float* w, float* dg, int64_t dg_fs, float* dd, int64_t dd_fs,
                          float* dw, float* dbias, void* stream);

/* ------------------------------------------------------------------------
 * Heads.  RGB_OFF.py:783-793,:844-847; Flow_OFF.py:867-876; basic_ops.py:12-46
 * ---------------------------------------------------------------------- */
/* All head tensors are channels-last: x[P, HW, ctot], slices are channel ranges [coff, coff+C).
 * out[p,c] = drop( mean_{hw} x[p, hw, x_coff+c] )   (global_pool RGB_OFF.py:262 + dropout :356) */
int offk_avgpool_drop_fwd(const float* x, int P, int C, int HW, int x_ctot, int x_coff, int drop_mode,
                          const uint8_t* keep_mask, uint64_t seed, const uint64_t* seed_dev, float drop_p, float keep_scale,
                          float* out, void* stream);
/* seed_dev (may be NULL) as in offk_stencil_t: the effective seed is seed + *seed_dev, read when the kernel runs.
 * offk_seed_set stores `value` into the device word. */
int offk_seed_set(uint64_t* state, uint64_t value, void* stream);
/* One head in ONE launch (SURVEY K6): global_pool -> dropout -> fc_action_motion* (-> ConsensusModule('avg') over the T
 * frame pairs of a clip): RGB_OFF.py:784-787, 790-793, 844-847; Flow_OFF.py:867-876; basic_ops.py:21-22.
 *   pooled[p, c]  = drop( mean_hw x[p, hw, x_coff + c] )                (written when non-NULL: the backward needs it)
 *   out[p, n]     = bias[n] + sum_c weight[n, c] * pooled[p, c]         weight [num_classes, C] row-major, exact fp32
 *   consensus_out[b, n] = mean_{t < T} out[b*T + t, n]                  (T > 1; NULL with T == 1: per-pair logits, RGB_OFF.py:860)
 * C % 4 == 0, C <= 1024, num_classes <= 128. */
int offk_head_fwd(const float* x, int P, int C, int HW, int x_ctot, int x_coff, int drop_mode, const uint8_t* keep_mask,
                  uint64_t seed, const uint64_t* seed_dev, float drop_p, float keep_scale, const float* weight,
                  const float* bias, int num_classes, int T, float* pooled, float* out, float* consensus_out, void* stream);
/* Backward of the above in two launches.  dout is [P / T, num_classes]: with T > 1 the consensus backward
 * (g.expand / T, basic_ops.py:30-31) is folded in, dfc(p, n) = dout[p / T, n] / T.
 *   dweight[n, c] += sum_p dfc(p, n) * pooled[p, c];  dbias[n] += sum_p dfc(p, n)                       (skipped when NULL)
 *   dx[p, hw, coff + c] = gate( dx_in + drop'( sum_n dfc(p, n) * weight[n, c] ) / HW )                   (skipped when dx NULL)
 *     dx_in = dx itself when accumulate != 0; gate = (act[same element] > 0) when act != NULL (ReLU' of the producer) */
int offk_head_bwd(const float* dout, int P, int C, int HW, int ctot, int coff, int drop_mode, const uint8_t* keep_mask,
                  uint64_t seed, const uint64_t* seed_dev, float drop_p, float keep_scale, const float* weight,
                  int num_classes, int T, const float* pooled, const float* act, int accumulate, float* dx,
                  float* dweight, float* dbias, void* stream);
/* 3x3 pool with ceil-mode output size between channel slices of channels-last tensors:
 *   x [n_img, H, W, x_ctot], channels [x_coff, x_coff + C)  ->  y [n_img, Ho, Wo, y_ctot], channels [y_coff, y_coff + C)
 *   Ho = ceil((H + 2 pad - 3) / stride) + 1, minus one if that last window would start at or past H + pad (the rule of
 *   F.max_pool2d / F.avg_pool2d with ceil_mode=True); likewise Wo.  pad <= 1.
 *   OFFK_POOL_MAX: max over the window elements inside the input (a window cut by the edge takes the max of the rest)
 *   OFFK_POOL_AVG: sum over the window elements inside the input / 9 (count_include_pad=True); every window must lie
 *                  inside the padded input, which holds for stride 1, pad 1
 * C, x_ctot, x_coff, y_ctot, y_coff multiples of 4, x and y 16-byte aligned.  Used for motion_pool_trans_28
 * (RGB_OFF.py:353,:783: max, stride 2, pad 0) and every pool of the BN-Inception extractor (RGB_OFF.py:43-263,362-594:
 * pool1 / pool2 and the stride-2 modules 3c / 4e: max, stride 2, pad 0; the normal modules: avg, stride 1, pad 1; 5b:
 * max, stride 1, pad 1). */
#define OFFK_POOL_MAX 0
#define OFFK_POOL_AVG 1
int offk_pool3_nhwc(const float* x, int n_img, int H, int W, int x_ctot, int x_coff, int C, int stride, int pad, int kind,
                    float* y, int y_ctot, int y_coff, void* stream);
/* ConsensusModule('avg', dim=1): out[b,:] = mean_t x[b,t,:]  (basic_ops.py:21-22) and its backward (:30-31) */
int offk_segment_mean_fwd(const float* x, int B, int T, int C, float* out, void* stream);
int offk_segment_mean_bwd(const float* dout, int B, int T, int C, float* dx, void* stream);
/* p[0..n) = 0 on `stream` (cudaMemsetAsync): zero-initialises split-K / atomic accumulation targets, e.g. the
 * gradient buffers before autograd of train_off.py:136-146 accumulates into them */
int offk_fill_zero(float* p, long long n, void* stream);
/* out = act > 0 ? grad : 0  (ReLU' as a stand-alone pass; n elements) */
int offk_relu_gate(const float* grad, const float* act, long long n, float* out, void* stream);
/* dst[p, dst_coff+c, :] = act[p, act_coff+c, :] > 0 ? src[p, src_coff+c, :] : 0  between channel slices of
 * [P, ctot, HW] buffers (ReLU' of motion_conv3_trans_14b, RGB_OFF.py:777-778, whose gradient arrives as a slice) */
int offk_gate_copy(const float* src, int src_ctot, int src_coff, const float* act, int act_ctot, int act_coff,
                   float* dst, int dst_ctot, int dst_coff, int P, int C, int HW, void* stream);
/* y[p, coff+c, :] += bias[c], then max(.,0) for c < relu_cols: finishes a split-K GEMM output slice */
int offk_bias_act(float* y, const float* bias, int P, int C, int HW, int ctot, int coff, int relu_cols,
                  void* stream);
/* dst[p, dst_coff+c, :] = act(a[p,c,:] + b[p,c,:])  -- sum_14b = relu(sum_14a + conv3_14b), RGB_OFF.py:779-780,
 * written straight into the 7-stage fusion buffer (cat, :832) */
int offk_add_relu_slice(const float* a, const float* b, float* dst, int dst_ctot, int dst_coff, int P, int C, int HW,
                        int relu, void* stream);

/* Conv weights: the reference's OIHW [cout,cin,kh,kw] <-> OHWI [cout,kh,kw,cin], the K order of the channels-last
 * implicit GEMM.  to_ohwi = 1: dst(OHWI) = src(OIHW) (before forward); 0: dst(OIHW) = src(OHWI);
 * 2: dst(OIHW) += src(OHWI) (weight gradients).
 * n (<= 16) weights in ONE launch, same to_ohwi for all (the OHWI -> OIHW accumulation of every KxK weight gradient
 * after the backward pass) */
typedef struct offk_permute {
  const float* src;
  float* dst;
  int32_t cout, cin, kh, kw;
} offk_permute_t;
int offk_permute_weight_batch(int n, const offk_permute_t* items, int to_ohwi, void* stream);

/* dst[i] = tf32 residual of src[i] = rn_tf32(src[i] - trunc_tf32(src[i])), i < n (n % 4 == 0, 16-byte aligned): the "lo" part
 * of the 3xTF32 split (OFFK_PREC_TF32X3) for operands that are known ahead of the GEMM -- the weights (offk_tgemm_t.b_lo_delta) */
int offk_tf32_residual(const float* src, float* dst, long long n, void* stream);

/* dst[i] = src[idx[i]], i < n.  One launch re-lays every conv weight of the step: OHWI copies for the forward
 * implicit GEMMs and [cin][kh][kw][cout] copies with flipped taps for the data-gradient GEMMs (autograd of
 * RGB_OFF.py:657-841); idx is built once on the host.  idx and dst 16-byte aligned. */
int offk_gather_copy(const float* src, const int32_t* idx, float* dst, long long n, void* stream);

/* dst[n, hw, c] = src[n, c, hw]: channels-last copy of an NCHW tensor.  Used for the 7x7 taps (inception_5a / 5b,
 * RGB_OFF.py:567,590): their 196-byte channel stride is not a legal TMA stride, so the unit's 1x1 conv and its weight
 * gradient read this copy through dense / im2col tensor maps instead. */
int offk_nchw_to_nhwc(const float* src, float* dst, int n_img, int C, int HW, void* stream);

/* dst[n, p, c'] = c' < c ? src[n, c', p] : 0, p < hw, c' < c_pad: the NCHW image batch of the BN-Inception extractor as a
 * channels-last tensor whose channel count c_pad (a multiple of 4: 4 for RGB, 12 for the 10-channel flow stack) gives the
 * stem conv 16-byte channel groups.  dst 16-byte aligned. */
int offk_image_to_nhwc(const float* src, float* dst, int n_img, int c, int hw, int c_pad, void* stream);

/* ------------------------------------------------------------------------
 * The training step around the path (train_off.py:72,133-151), on the flat parameter / gradient buffers.
 * ---------------------------------------------------------------------- */
/* nn.CrossEntropyLoss (mean over the P rows) of logits [P, C] against the clip labels repeated per frame pair
 * (train_off.py:133: target.unsqueeze(1).repeat(1, num_seg-1).view(-1)): label of row p = target[p / repeat].
 * loss_accum (may be NULL) += the loss; dlogits (may be NULL) = grad_scale * dLoss/dlogits.  Several heads may
 * accumulate into the same loss_accum (train_off.py:136-146 sums three CE terms by calling backward three times). */
int offk_ce_loss_fwd_bwd(const float* logits, const long long* target, int P, int C, int repeat, float grad_scale,
                         float* loss_accum, float* dlogits, void* stream);
/* sumsq_accum += sum_i g[i]^2 (double; the caller zeroes it): the squared global norm of clip_grad_norm (train_off.py:149) */
int offk_grad_sumsq(const float* g, long long n, double* sumsq_accum, void* stream);
/* clip_grad_norm(params, max_norm) + optim.Adam(lr, betas, weight_decay).step() (train_off.py:72,149-151) in ONE pass over
 * the element ranges [range_lo[k], range_hi[k]) (multiples of 4) of the flat buffers p, g, m (exp_avg), v (exp_avg_sq):
 *   coef = min(1, max_norm / (sqrt(*sumsq) + 1e-6))     (sumsq == NULL or max_norm <= 0: no clipping)
 *   g' = coef * g + weight_decay * p;  m = b1 m + (1-b1) g';  v = b2 v + (1-b2) g'^2
 *   p -= lr / (1 - b1^step) * m / (sqrt(v) / sqrt(1 - b2^step) + eps)                      (step counts from 1)
 * The norm is read from device memory: no host synchronisation between backward and the update.  Ranges let the caller
 * skip parameters that have no gradient in the reference (fc_action_motion_28, RGB_OFF.py:787,860). */
#define OFFK_ADAM_MAX_RANGES 8
int offk_clip_adam_step(float* p, const float* g, float* m, float* v, const long long* range_lo, const long long* range_hi,
                        int n_ranges, float lr, float beta1, float beta2, float eps, float weight_decay, int step,
                        float max_norm, const double* sumsq, void* stream);

/* keep decision of OFFK_DROP_SEED for element `idx` (host mirror for tests): 1 = keep */
int offk_drop_keep_host(uint64_t seed, uint64_t idx, float drop_p);

#ifdef __cplusplus
}
#endif
#endif /* OFFK_H_ */
