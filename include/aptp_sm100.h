/*
 * aptp_sm100.h -- C ABI of libaptp_sm100.so: the B200 (sm_100a) kernels behind the APTP gated
 * SD-2.1 U-Net denoising step and its router (reference: rezashkv/diffusion_pruning).
 *
 * Conventions
 *   - every entry point returns 0 (APTP_OK) or a negative status; aptp_last_error() gives the text;
 *   - no allocation, no implicit synchronisation: all pointers are device pointers owned by the caller
 *     (PyTorch), work is enqueued on `stream` (a cudaStream_t passed as void*);
 *   - activations are NHWC / token-major bf16: a [B,C,H,W] reference tensor is stored as rows
 *     (b*H*W + y*W + x) of C contiguous channels, so conv-as-GEMM, Linear and the [B,HW,C] token
 *     view used by the reference (pdm/models/unet/blocks.py:1235, :1306) are the same memory;
 *   - samples are bucketed by architecture code ("expert"); a *segment* describes one bucket of a
 *     layer: its row range, kept output columns, kept K chunks and where its compacted weights live.
 *
 * Each function cites the reference code it replaces (paths relative to the reference repo).
 */
#ifndef APTP_SM100_H
#define APTP_SM100_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define APTP_ABI_VERSION 2

/* library / diagnostics */
int aptp_version(void);
const char* aptp_last_error(void);
/* returns 1 if a pipelined kernel hit an mbarrier timeout since the last call (and clears it); syncs `stream`. */
int aptp_check_abort(void* stream);
/* non-blocking: returns 1 if the flag copy enqueued by the previous call shows a timeout (and clears it), then enqueues
 * a new 4-byte copy behind the work on `stream`. Called by every forward / step of the host code (no host sync). */
int aptp_poll_abort(void* stream);

/* ------------------------------------------------------------------------------------------------
 * K1  grouped, expert-bucketed GEMM / implicit-GEMM conv on tcgen05 + TMEM fed by TMA.
 *     out[rows, n] = epilogue( sum_k A[rows, k] * W[w_row_off + n, k] )
 * replaces: F.conv2d / F.linear call sites of ResnetBlock2DWidth(Depth)Gated.forward
 *   (pdm/models/unet/blocks.py:331,:337,:362,:366,:537,:568,:572), GatedAttention projections
 *   (blocks.py:228-240,:266-268), GEGLUGated.forward (blocks.py:41-50), FeedForward.net[2],
 *   Transformer2DModel.proj_in/out (blocks.py:1239-1243,:1301-1305), conv_in/conv_out and the
 *   down/up-sampler convs (pdm/models/unet/unet_2d_conditional.py:1614,:1721), and -- through the
 *   compacted per-expert weight blocks -- the prune() family (blocks.py:52-67,:121-129,:153-187,
 *   :424-465).
 * ---------------------------------------------------------------------------------------------- */
typedef struct aptp_gemm_seg {
  int32_t row_begin; /* first output row of this expert bucket                                   */
  int32_t row_end;   /* one past its last output row (rows >= row_end are never written)          */
  int32_t n_valid;   /* kept output columns (GEGLU: kept *output* columns, i.e. h columns)        */
  int32_t n_store;   /* columns [n_valid, n_store) are written as zeros (K padding for consumer)  */
  int32_t k_chunks;  /* 64-wide K chunks per tap that carry kept input channels                   */
  int32_t w_row_off; /* first row of this bucket's block in the packed weight matrix              */
  int32_t vec_off;   /* offset of this bucket's bias (floats) in `bias`                           */
  int32_t tab_off;   /* offset of this bucket's 9 x n border table (floats) in `border_tab`       */
  int32_t out_col_off; /* output / residual column of this bucket's column 0 (fused q|k|v blocks)   */
  int32_t w2_row_off;  /* first row of this bucket's block in `w2` (second operand pair, a2 / w2)     */
  int32_t pad1, pad2;
} aptp_gemm_seg;

typedef struct aptp_gemm_tile {
  int32_t seg;    /* index into segs                                                              */
  int32_t m_base; /* linear: first row; conv: linear index of the top-left output pixel of the box */
  int32_t n0;     /* first packed weight row / accumulator column block of this tile              */
  int32_t flags;  /* APTP_TILE_* in bits 0..7; bits 8..15: tile width / 32 when the bucket's column tiles are
                     narrower than bn (balanced tiles; 0 = bn wide; not for GEGLU)                 */
} aptp_gemm_tile;
/* Tiles are consumed in PAIRS by a cluster of two CTAs that share (multicast) the weight tile: n_tiles is
 * even and tiles[2i], tiles[2i+1] have the same seg and n0 and different m_base. A bucket with an odd
 * number of row tiles is padded with a placeholder that repeats its partner's m_base and stores nothing. */
enum {
  APTP_TILE_PLACEHOLDER = 1,
  /* A-stationary tile lists (a_stat_chunks > 0): CTA pair c of the S = min(runs, aptp_gemm_max_pairs()) pairs in the
   * grid consumes entries c, c + S, c + 2S, ...; the host orders them so that every pair sees all N tiles of one pair
   * of row tiles back to back. The first entry of such a run loads the A row tile (A_FIRST), the last one releases it
   * (A_LAST); SKIP entries pad the shorter sequences and do nothing. */
  APTP_TILE_A_FIRST = 2,
  APTP_TILE_A_LAST = 4,
  APTP_TILE_SKIP = 8
};

enum { APTP_A_LINEAR = 0, APTP_A_CONV3X3 = 1, APTP_A_CONV3X3_S2 = 2 };
enum { APTP_OUT_BF16 = 0, APTP_OUT_F32 = 1, APTP_OUT_F32_NCHW = 2 };
enum {
  APTP_EPI_GEGLU = 1,      /* tile columns are [bn/2 h | bn/2 g]; out = h * gelu_erf(g)            */
  APTP_EPI_SILU = 2,       /* out = silu(out) (time-embedding MLP)                                 */
  APTP_EPI_GN_STATS = 4,   /* per-channel (sum, sumsq) partials of the stored fp32 rows, see gn_stats */
  APTP_EPI_RES_F32 = 8,    /* `residual` holds fp32 rows (fp32 residual stream); needs APTP_OUT_F32 */
  APTP_EPI_LN_FOLD = 16    /* LayerNorm of the A rows folded into this GEMM (see ln_* below)         */
};

typedef struct aptp_gemm_args {
  /* A operand: bf16 activations */
  const void* a;
  int32_t a_mode;  /* APTP_A_*                                                                     */
  int32_t a_ld;    /* elements between consecutive rows / pixels                                   */
  int32_t a_k;     /* addressable channels per pixel (tensor-map extent; reads beyond are zero)    */
  int64_t a_rows;  /* linear: rows; conv: batch*H*W input pixels                                   */
  int32_t batch, H, W; /* conv: INPUT spatial size                                                 */
  /* B operand: packed bf16 weights [w_rows, w_ld], K-major; conv K index = tap*k_tap_pitch + c    */
  const void* w;
  int64_t w_rows;
  int32_t w_ld;
  int32_t k_tap_pitch;
  /* output */
  void* out;
  int32_t out_ld;
  int32_t out_mode; /* APTP_OUT_*                                                                  */
  /* tile shape: M tile is 128 rows = box bw x bh x bb output pixels (linear: 128 x 1 x 1)         */
  int32_t bn;       /* accumulator columns per tile: multiple of 32, 32..256                       */
  int32_t bw, bh, bb;
  /* epilogue operands (any may be NULL) */
  const float* bias;      /* [.. vec_off + col]                                                    */
  const float* rowvec;    /* per-sample vector: rowvec[sample*rowvec_ld + col] (time embedding)    */
  int32_t rowvec_ld;
  int32_t rows_per_sample;
  const void* residual;   /* bf16 [rows, res_ld] (fp32 with APTP_EPI_RES_F32), added after everything else; may alias out */
  int32_t res_ld;
  const float* gate;      /* soft gates: out *= gate[sample*gate_ld + col/gate_group]              */
  int32_t gate_ld, gate_group;
  const float* border_tab; /* conv2 of a width-compacted ResNet: contribution of the pruned input
                              channels, which the *gated* reference still feeds as silu(beta_c)
                              (SURVEY Appendix D-1); [tab_off + (ycls*3+xcls)*tab_ld + col]        */
  int32_t tab_ld;
  /* APTP_EPI_GN_STATS (needs APTP_OUT_F32): GroupNorm statistics of the tensor this GEMM writes, gathered in its
   * epilogue so the consumer's statistics pass over HBM disappears. Every (tile, 32-row quadrant) writes the column
   * sums / sums of squares of its 32 rows x N columns:
   *   gn_stats   [ (sample * gn_blocks + blk) * gn_ld + out_col_off + col ] = sum over the 32 rows
   *   gn_stats_sq[ same index ]                                              = sum of squares
   * blk = (tile index inside the sample) * 4 + quadrant, gn_blocks = rows_per_sample / 32. Requires
   * rows_per_sample % 128 == 0 and, for conv tiles, a box inside one image (bb == 1). No atomics: every entry has
   * one writer; aptp_groupnorm_stats_from_partials reduces them per (sample, group) in a fixed order. */
  float* gn_stats;
  int32_t gn_ld;          /* floats per partial row (>= channels of the output tensor)              */
  int32_t gn_blocks;      /* 32-row blocks per sample                                             */
  int32_t flags;          /* APTP_EPI_*                                                            */
  /* schedule (device memory) */
  const aptp_gemm_seg* segs;
  int32_t n_segs;
  const aptp_gemm_tile* tiles;
  int32_t n_tiles;
  /* LayerNorm folded into the GEMM (APTP_EPI_LN_FOLD; replaces BasicTransformerBlock.norm1/2/3, blocks.py:782,:808-810,
   * :821): `a` holds the RAW rows x, `w` holds W*gamma, `bias` holds W@beta (+ the layer's own bias) and
   *   out[row, n] = rstd[row] * (acc[row, n] - mean[row] * ln_colsum[vec_off + n]) + bias[vec_off + n]
   * where ln_colsum[n] = sum_k w[n, k] (of the bf16-rounded packed weights) and ln_rowstats[row] = (mean, rstd) of the
   * row (float2, from aptp_ln_rowstats). The (sum, sumsq) partials behind them are written by the GEMM that PRODUCED x:
   * rowstat_out[row * rowstat_chunks + (out_col_off + col) / 32] (of the values it stores, bf16 output only).
   * Deterministic (no atomics). */
  const float* ln_colsum;
  const float* ln_rowstats;  /* float2 per row: (mean, rstd) */
  int32_t ln_reserved0;
  int32_t ln_reserved1;
  float ln_reserved2;
  float* rowstat_out;        /* float2 per (row, chunk) */
  int32_t rowstat_chunks;
  float* gn_stats_sq;        /* APTP_EPI_GN_STATS: the sum-of-squares plane (same indexing as gn_stats) */
  int32_t a_stat_chunks;     /* > 0: A-stationary tile list (see APTP_TILE_A_FIRST); = max k_chunks over the segments,
                                at most 6 (K <= 384), linear layers only                                          */
  int32_t a_stat_pairs;      /* the number S of CTA pairs the A-stationary tile list was laid out for              */
  /* Second operand pair accumulated into the SAME tiles (APTP_A_CONV3X3 only): out += A2[pixel, :] * W2[n, :]^T, a 1x1
   * conv over a second NHWC tensor of the same batch / H / W -- ResnetBlock2D.conv_shortcut over the (concatenated)
   * block input (blocks.py:367-369), so the shortcut costs no launch, no fp32 round trip and no residual read. W2 is
   * [>= n, a2_k] bf16 with row pitch w2_ld, indexed by the output column (not compacted); its bias is expected in
   * `bias`. NULL a2: none. Honoured by the halo-tile scheme (8 x 16-pixel boxes, reductions >= 1280); otherwise
   * aptp_grouped_gemm_fwd returns APTP_ERR_UNSUPPORTED and the caller launches the 1x1 conv itself. */
  const void* a2;
  int32_t a2_ld;
  int32_t a2_k;
  const void* w2;
  int64_t w2_rows;
  int32_t w2_ld;
} aptp_gemm_args;

int aptp_grouped_gemm_fwd(const aptp_gemm_args* args, void* stream);
/* CTA pairs of the GEMM kernel that are co-resident on this device (the grid is 2 * min(pairs of tiles, this)). */
int aptp_gemm_max_pairs(void);

/* ------------------------------------------------------------------------------------------------
 * K2  HBM-bound fused normalisation / gate / residual kernels.
 * ---------------------------------------------------------------------------------------------- */
/* GroupNorm statistics over NHWC rows (two sources = fused torch.cat of an up-block input); x_f32 != 0: the
 * sources are fp32 rows (the fp32 residual stream between blocks), else bf16.
 * replaces: the reduction half of nn.GroupNorm at blocks.py:299,:353,:505,:559, Transformer2DModel.norm
 * (blocks.py:1227) and conv_norm_out (unet_2d_conditional.py:1719).
 * stats[sample][group] = (sum, sumsq) in fp32, OVERWRITTEN (no zeroing needed). The reduction is deterministic:
 * fixed-order partial sums per CTA, merged in chunk order by the last CTA of each sample. `workspace` (device,
 * 16-byte aligned, >= aptp_groupnorm_stats_workspace(batch, hw, stats_groups) bytes) must have its first
 * 4*batch bytes zero before the FIRST call; every call leaves them zero. One workspace per stream. */
int64_t aptp_groupnorm_stats_workspace(int32_t batch, int32_t hw, int32_t stats_groups);
int aptp_groupnorm_stats(const void* x0, int32_t c0, int32_t ld0, const void* x1, int32_t c1, int32_t ld1,
                         int32_t x_f32, int32_t batch, int32_t hw, int32_t group_size,
                         const int32_t* sample_channels, float* stats, int32_t stats_groups, void* workspace,
                         int64_t workspace_bytes, void* stream);
/* stats[sample][group] = (sum, sumsq) from the per-channel partials that GEMM epilogues wrote (APTP_EPI_GN_STATS):
 * up to two sources (the halves of an up-block torch.cat) with their own partial planes [batch][blocks][ld]; group g
 * covers concatenated channels [g*group_size, (g+1)*group_size). Fixed summation order (deterministic). */
int aptp_groupnorm_stats_from_partials(const float* sum0, const float* sq0, int32_t c0, int32_t ld0, const float* sum1,
                                       const float* sq1, int32_t c1, int32_t ld1, int32_t blocks, int32_t batch,
                                       int32_t group_size, const int32_t* sample_channels, float* stats,
                                       int32_t stats_groups, void* stream);
/* y = [silu]( (x*g - mean)*rstd*gamma + beta ) written bf16 with row pitch ldy; channels in
 * [c_valid, c_store) are written as zeros. `sample_seg[b]` selects the per-expert compacted
 * gamma/beta block (offset sample_seg[b]*affine_ld) and c_valid (sample_channels[b]).
 * `gate` (optional, fp32 [batch, gate_ld]) is the soft width gate applied *before* the norm
 * (blocks.py:345-353): with hard gates the engine compacts instead. x_f32 as above. */
int aptp_groupnorm_apply(const void* x0, int32_t c0, int32_t ld0, const void* x1, int32_t c1, int32_t ld1,
                         int32_t x_f32, void* y, int32_t ldy, int32_t batch, int32_t hw, int32_t group_size,
                         float eps, const float* stats, int32_t stats_groups, const float* gamma,
                         const float* beta, int32_t affine_ld, const int32_t* sample_seg,
                         const int32_t* sample_channels, const float* gate, int32_t gate_ld, int32_t silu,
                         void* stream);
/* The same pass additionally writes `raw_out` (bf16 rows, pitch raw_ld, may be NULL): the UN-normalised input converted
 * to bf16 with both sources concatenated -- the A operand of ResnetBlock2D's 1x1 conv_shortcut over
 * torch.cat([hidden_states, res_hidden_states], 1) (blocks.py:367-369) -- so the fp32 stream is read once for both. */
int aptp_groupnorm_apply_raw(const void* x0, int32_t c0, int32_t ld0, const void* x1, int32_t c1, int32_t ld1,
                             int32_t x_f32, void* y, int32_t ldy, int32_t batch, int32_t hw, int32_t group_size,
                             float eps, const float* stats, int32_t stats_groups, const float* gamma,
                             const float* beta, int32_t affine_ld, const int32_t* sample_seg,
                             const int32_t* sample_channels, const float* gate, int32_t gate_ld, int32_t silu,
                             void* raw_out, int32_t raw_ld, void* stream);
/* LayerNorm over the channel dim of [rows, C] bf16 (eps 1e-5, affine); replaces
 * BasicTransformerBlock.norm1/2/3 (blocks.py:782,:808-810,:821). row_active (optional, per sample)
 * skips depth-dropped samples. */
int aptp_layernorm(const void* x, int32_t ldx, void* y, int32_t ldy, int64_t rows, int32_t C, float eps,
                   const float* gamma, const float* beta, const uint8_t* sample_active,
                   int32_t rows_per_sample, void* stream);
/* (mean, rstd) per row [rows] float2 from the per-chunk (sum, sumsq) partials a GEMM epilogue wrote (rowstat_out of
 * aptp_gemm_args): the row statistics of the LayerNorm that APTP_EPI_LN_FOLD folds into the consuming GEMM. */
int aptp_ln_rowstats(const float* partial, int32_t chunks, int64_t rows, int32_t C, float eps, float* out,
                     const uint8_t* sample_active, int32_t rows_per_sample, void* stream);
/* out = (1-d)*x + d*y per sample (DepthGate.forward, pdm/models/unet/gates.py:36-42), bf16 rows. */
int aptp_depth_lerp(const void* x, int32_t ldx, const void* y, int32_t ldy, void* out, int32_t ldo,
                    int64_t rows, int32_t C, const float* d, int32_t rows_per_sample, void* stream);
/* dst[rows, :C] = src[rows, :C] for the samples with sample_mask[b] != 0 (NULL = all): identity path
 * of depth-dropped blocks (blocks.py:497-498,:1190-1194) and torch.cat of up-block skips. */
int aptp_copy_rows(const void* src, int32_t lds, void* dst, int32_t ldd, int64_t rows, int32_t C,
                   const uint8_t* sample_mask, int32_t rows_per_sample, void* stream);
/* nearest x2 upsample NHWC (diffusers Upsample2D: F.interpolate(scale_factor=2, mode="nearest")). */
int aptp_upsample2x(const void* src, void* dst, int32_t batch, int32_t H, int32_t W, int32_t C, void* stream);
/* fp32-residual-stream variants (the tensors between ResNet / transformer blocks are kept in fp32 so that the
 * residual sums of unet_2d_conditional.py:1629-1715 are not re-rounded to bf16 at every block; GEMM A operands
 * stay bf16): row copy with conversion (src / dst each bf16 or fp32), DepthGate lerp on fp32 rows (out may alias
 * y), nearest x2 upsample from fp32 or bf16 rows to bf16 rows. */
int aptp_copy_rows_cvt(const void* src, int32_t src_f32, int32_t lds, void* dst, int32_t dst_f32, int32_t ldd,
                       int64_t rows, int32_t C, const uint8_t* sample_mask, int32_t rows_per_sample, void* stream);
int aptp_depth_lerp_f32(const float* x, int32_t ldx, const float* y, int32_t ldy, float* out, int32_t ldo,
                        int64_t rows, int32_t C, const float* d, int32_t rows_per_sample, void* stream);
int aptp_upsample2x_cvt(const void* src, int32_t src_f32, void* dst, int32_t batch, int32_t H, int32_t W, int32_t C,
                        void* stream);
/* NCHW fp32 sample -> im2col rows [B*H*W, 64] bf16 (K = 9*Cin zero-padded to 64) for conv_in. */
int aptp_im2col_input(const float* sample_nchw, void* dst, int32_t batch, int32_t Cin, int32_t H, int32_t W,
                      void* stream);
/* Timesteps(320, flip_sin_to_cos=True, freq_shift=0): emb[b] = [cos(t f_k), sin(t f_k)] as bf16. */
int aptp_timestep_embedding(const float* t, void* dst, int32_t batch, int32_t dim, void* stream);
/* fp32 -> bf16 cast (text embeddings), plain elementwise silu over bf16. */
int aptp_cast_f32_bf16(const float* src, void* dst, int64_t n, void* stream);
int aptp_silu_bf16(const void* src, void* dst, int64_t n, void* stream);
/* Fused classifier-free-guidance combine + DDIM update (eta 0) of the sampling loop
 * (pdm/pipelines/pruning_pipelines.py:805-814; diffusers DDIMScheduler.step, SURVEY Appendix B):
 * pred = [uncond | cond] noise predictions (2n floats), x / x_out = latents (n floats); alpha_* are
 * alphas_cumprod at the current / previous timestep. */
int aptp_cfg_ddim_step(const float* pred, const float* x, float* x_out, int64_t n, float guidance, float alpha_t,
                       float alpha_prev, int32_t v_prediction, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K3  flash-style attention on tcgen05 with per-sample kept-head lists.
 * replaces: HeadGatedAttnProcessor2.__call__ head gating + F.scaled_dot_product_attention
 * (blocks.py:245-262). q/k/v are bf16 [tokens, ld] with head h at columns [h*64, h*64+64) of the
 * *compacted* projection; sample_heads[b] = kept heads of sample b (its bucket); samples with 0 heads
 * are skipped. out has the same compacted layout.
 * ---------------------------------------------------------------------------------------------- */
int aptp_attention_fwd(const void* q, int32_t ldq, const void* k, int32_t ldk, const void* v, int32_t ldv,
                       void* out, int32_t ldo, int32_t batch, int32_t n_q, int32_t n_kv,
                       const int32_t* sample_heads, int32_t max_heads, float scale, float* lse2, void* stream);
/* lse2 (optional, may be NULL): [batch, max_heads, n_q] fp32, log2-domain log-sum-exp of the scaled scores,
 * consumed by aptp_attention_bwd. */
/* Backward (K5): dq, dk, dv of the same attention (compacted head layout as the forward); `o` is the forward
 * output, `dout` its gradient, delta is scratch [batch, max_heads, n_q] (rowsum(dout*o), written here).
 * Two tcgen05 kernels: Q-stationary (dq) and KV-stationary (dk, dv). */
int aptp_attention_bwd(const void* q, int32_t ldq, const void* k, int32_t ldk, const void* v, int32_t ldv,
                       const void* o, int32_t ldo, const void* dout, int32_t lddo, const float* lse2, float* delta,
                       void* dq, int32_t lddq, void* dk, int32_t lddk, void* dv, int32_t lddv, int32_t batch,
                       int32_t n_q, int32_t n_kv, const int32_t* sample_heads, int32_t max_heads, float scale,
                       void* stream);

/* ------------------------------------------------------------------------------------------------
 * K4  router: fused Gumbel-sigmoid gate, width/depth normalisation, cosine scores, Sinkhorn, argmax.
 * ---------------------------------------------------------------------------------------------- */
/* gumbel_sigmoid_trick (pdm/models/vq/quantizer.py:196-215 + pdm/utils/estimation_utils.py:5-64):
 * width slices sigma((z + G + base)/T) with the all-zero fix-up (estimation_utils.py:23-31), depth
 * columns through softmax/cumsum/flip/logit (estimation_utils.py:49-64) scattered by depth_order.
 * `u` are the uniforms the reference draws on the CPU (depth [B,n_depth] first, then the width
 * slices in order), laid out [B, n_width + n_depth] in arch-vector column order. */
int aptp_gumbel_gate_fwd(const float* z, const float* u, float* out, int32_t batch, int32_t n_width,
                         int32_t n_depth, const int32_t* width_starts, int32_t n_width_gates,
                         const int32_t* depth_order, float temperature, float base, int32_t non_zero_width,
                         void* stream);
/* backward of aptp_gumbel_gate_fwd w.r.t. z (dl = dy*y(1-y)/T, estimation_utils.py:40-41; depth through
 * logit/flip/cumsum/softmax, estimation_utils.py:50-56, and the depth_order scatter quantizer.py:205-206). */
int aptp_gumbel_gate_bwd(const float* z, const float* u, const float* dy, float* dz, int32_t batch, int32_t n_width,
                         int32_t n_depth, const int32_t* depth_order, float temperature, float base, void* stream);
/* width_depth_normalize (quantizer.py:233-250) + L2 normalise (quantizer.py:266-267,:326-327):
 * out[b,:] = v/||v|| (or v when l2_normalize = 0), v = (width slices of depth-gated blocks * their depth gate, hard_concrete
 * elsewhere) * sqrt(template) [* macs_template]. col_depth[c] = arch column of the depth gate that
 * multiplies column c, or -1. */
int aptp_arch_normalize(const float* gates, float* out, int32_t batch, int32_t dim, const int32_t* col_depth,
                        const float* col_scale, int32_t l2_normalize, void* stream);
/* backward of the l2_normalize=0 form (hard_concrete straight-through; product rule on depth-gated slices). */
int aptp_arch_normalize_bwd(const float* gates, const float* dy, float* dx, int32_t batch, int32_t dim,
                            const int32_t* col_depth, const float* col_scale, void* stream);
/* scores = A @ C^T  ([B,dim] x [K,dim]) in fp32 and argmax per row (quantizer.py:264-271). */
int aptp_route_cosine(const float* a_norm, const float* codes_norm, float* scores, int64_t* indices,
                      int32_t batch, int32_t dim, int32_t n_codes, void* stream);
/* Sinkhorn OT assignment (quantizer.py:274-340). Phase API so that the 4 marginal all-reduces of
 * distributed_sinkhorn (quantizer.py:285,:291) run as NCCL calls on the same stream between phases:
 *   phase 0: Q = exp(S/eps); partial[0] = sum(Q)                       -> all-reduce partial[0:1]
 *   phase 1 (x iters): Q /= total (first) ; row sums -> partial[0:K]   -> all-reduce partial[0:K]
 *   phase 2: Q /= rowsum*K ; column-normalise ; /B
 *   phase 3: argmax per sample.
 * aptp_route_sinkhorn runs all phases for the single-process case. Marginals accumulate in fp64. */
int aptp_sinkhorn_phase(int32_t phase, float* Q, const float* scores, double* partial, int64_t* indices,
                        int32_t batch_local, int32_t batch_global, int32_t n_codes, float epsilon,
                        int32_t first_iter, void* stream);
int aptp_route_sinkhorn(const float* scores, float* Q, double* partial, int64_t* indices, int32_t batch,
                        int32_t n_codes, float epsilon, int32_t iterations, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K5  backward of the gated ops (SURVEY Appendix G). The U-Net is frozen during pruning
 * (pdm/models/unet/unet_2d_conditional.py:2118-2122): only activation gradients (bf16) and
 * per-(sample, gate) reductions (fp32, accumulated with atomics into caller-zeroed buffers) exist.
 * dgrad GEMMs / convs reuse aptp_grouped_gemm_fwd with transposed (conv: tap-flipped) packed weights.
 * ---------------------------------------------------------------------------------------------- */
/* y = gate[b, c/group] * u over [batch*hw, C] (WidthGate on q,k,v: blocks.py:250-255; gates.py:15-21) */
int aptp_scale_cols_fwd(const void* u, int32_t ldu, void* y, int32_t ldy, int32_t batch, int32_t hw, int32_t C,
                        const float* gate, int32_t gate_ld, int32_t group, void* stream);
/* du = gate * dy ; dgate[b,k] += sum_{pixels, c in k} dy * u */
int aptp_scale_cols_bwd(const void* u, int32_t ldu, const void* dy, int32_t lddy, void* du, int32_t lddu, int32_t batch,
                        int32_t hw, int32_t C, const float* gate, int32_t gate_ld, int32_t group, float* dgate,
                        void* stream);
/* GEGLUGated.forward (blocks.py:41-50) on the un-packed projection hg = [h | gate] (training form):
 * out = (g h) * gelu_erf(g gate); backward writes d(hg) and accumulates dgate. gate may be NULL. */
int aptp_geglu_fwd(const void* hg, int32_t ld, void* out, int32_t ldo, int32_t batch, int32_t hw, int32_t inner,
                   const float* gate, int32_t gate_ld, int32_t group, void* stream);
int aptp_geglu_bwd(const void* hg, int32_t ld, const void* df, int32_t lddf, void* dhg, int32_t lddhg, int32_t batch,
                   int32_t hw, int32_t inner, const float* gate, int32_t gate_ld, int32_t group, float* dgate,
                   void* stream);
/* backward of aptp_groupnorm_apply (GroupNorm [+ width gate before, + SiLU after]; blocks.py:345-359):
 * dx (+)= ..., dgate[b, group] += sum dxg * x. `stats` are the forward (sum, sumsq); bstats is scratch
 * [batch, stats_groups, 2] (zeroed here). */
int aptp_groupnorm_bwd(const void* x, int32_t ldx, const void* da, int32_t ldda, void* dx, int32_t lddx,
                       int32_t accumulate, int32_t batch, int32_t hw, int32_t C, int32_t group_size, float eps,
                       const float* stats, int32_t stats_groups, const float* gamma, const float* beta,
                       const float* gate, int32_t gate_ld, int32_t silu, float* bstats, float* dgate, void* stream);
/* backward of aptp_layernorm w.r.t. x: dx (+)= rstd (dy gamma - mean(.) - xh mean(. xh)) */
int aptp_layernorm_bwd(const void* x, int32_t ldx, const void* dy, int32_t lddy, void* dx, int32_t lddx,
                       int32_t accumulate, int64_t rows, int32_t C, float eps, const float* gamma, void* stream);
/* DepthGate backward (gates.py:36-42): dy = d dout ; dx (+)= (1-d) dout ; dd[b] += sum dout (y - x) */
int aptp_depth_lerp_bwd(const void* dout, int32_t lddo, const void* x, int32_t ldx, const void* y, int32_t ldy,
                        void* dy, int32_t lddy, void* dx, int32_t lddx, int32_t accumulate, int32_t batch, int32_t hw,
                        int32_t C, const float* d, float* dd, void* stream);
/* dst += src (gradient fan-in of skips / residual branches) */
int aptp_add_rows(const void* src, int32_t lds, void* dst, int32_t ldd, int64_t rows, int32_t C, void* stream);
/* backward of aptp_upsample2x; and the zero-insertion that turns the stride-2 conv dgrad into a stride-1 conv
 * of the tap-flipped weights (H, W = output size of the forward conv). */
int aptp_upsample2x_bwd(const void* dy, void* dx, int32_t batch, int32_t H, int32_t W, int32_t C, void* stream);
int aptp_zero_insert2x(const void* src, void* dst, int32_t batch, int32_t H, int32_t W, int32_t C, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K6  loss front/back end of the pruning train step (SURVEY 8f rank 2), one HBM pass each.
 * ------------------------------------------------------------------------------------------------ */
/* DDIMScheduler.add_noise + get_velocity (pdm/training/trainer.py:1121-1123, :1181): noisy = sqrt(acp[t]) x0 +
 * sqrt(1-acp[t]) n; target = sqrt(acp[t]) n - sqrt(1-acp[t]) x0 (v_prediction) or n (epsilon). fp32 [batch,
 * per_sample]; timesteps int64 [batch]; sqrt_acp / sqrt_1m_acp = fp32 tables over the train timesteps; target may
 * be NULL. */
int aptp_add_noise_velocity(const float* latents, const float* noise, const int64_t* timesteps, const float* sqrt_acp,
                            const float* sqrt_1m_acp, float* noisy, float* target, int32_t batch, int32_t per_sample,
                            int32_t v_prediction, void* stream);
/* Block-distillation MSE (trainer.py:1220-1225) between two bf16 NHWC row tensors: partial[i] (fp64, i <
 * n_partial, every slot written) sums to sum((a-b)^2); the caller divides by the element count. */
int aptp_mse_rows_fwd(const void* a, int32_t lda, const void* b, int32_t ldb, int64_t rows, int32_t C, double* partial,
                      int32_t n_partial, void* stream);
/* da = coef[0] * scale * (a - b) as bf16 rows (coef: device scalar = upstream gradient, scale = 2 / numel). */
int aptp_mse_rows_bwd(const void* a, int32_t lda, const void* b, int32_t ldb, void* da, int32_t ldda, int64_t rows,
                      int32_t C, const float* coef, float scale, void* stream);
/* DDPM (min-SNR weighted) + distillation MSE on the fp32 predictions (trainer.py:1197-1218): partial[(b * chunks +
 * c) * 2 + {0, 1}] = sums of (pred-target)^2 and (pred-teacher)^2 over chunk c of sample b. */
int aptp_pred_losses_fwd(const float* pred, const float* target, const float* teacher, int32_t batch, int32_t per_sample,
                         int32_t chunks, double* partial, void* stream);
/* dpred = 2 / (batch * per_sample) * (g[0] * weight[b] * (pred-target) + g[1] * (pred-teacher)); weight may be NULL
 * (plain mean); g = device [2] upstream gradients of the two losses. */
int aptp_pred_losses_bwd(const float* pred, const float* target, const float* teacher, const float* weight,
                         const float* g, float* dpred, int32_t batch, int32_t per_sample, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K7  closed-form MAC accounting on the [B, 1620] gate matrix (SURVEY 8f rank 3, Appendix F).
 * replaces: UNet2DConditionModelGated.calc_macs tree walk (unet_2d_conditional.py:2124-2163 and the per-block
 * calc_macs methods, blocks.py:103-119 ... :1373-1413) with its hard_concrete calls (estimation_utils.py:67-75).
 * ------------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t col;    /* first column of this width gate in the gate matrix */
  int32_t width;  /* number of columns */
  double macs;    /* prunable MACs that scale with the gate's kept ratio (op_counter.py constants) */
} aptp_macs_gate;
typedef struct {
  int32_t first_gate, n_gates; /* its width gates (contiguous in get_structure order) */
  int32_t depth_col;           /* column of its depth gate, -1 if none */
  int32_t reserved;
  double fixed;                /* non-prunable MACs of the sub-block (total - prunable) */
} aptp_macs_sub;
/* cur_prunable[b], cur_total[b] (fp32 [batch]) = calc_macs()['cur_prunable_macs' / 'cur_total_macs'] for gate row b;
 * fixed_total = MACs outside the gated sub-blocks. Gates are thresholded at 0.5 (hard_concrete). */
int aptp_macs_ratio_fwd(const float* arch, int32_t ld, int32_t batch, const aptp_macs_gate* gates, int32_t n_gates,
                        const aptp_macs_sub* subs, int32_t n_subs, double fixed_total, float* cur_prunable,
                        float* cur_total, void* stream);
/* Straight-through gradient of cur_prunable to every gate column: darch[b, :dim] = dcur_prunable[b] * d cur_prunable[b]
 * / d arch[b, :] (cur_total carries none, as in the reference's .detach()). */
int aptp_macs_ratio_bwd(const float* arch, int32_t ld, int32_t batch, const aptp_macs_gate* gates, int32_t n_gates,
                        const aptp_macs_sub* subs, int32_t n_subs, const float* dcur_prunable, float* darch, int32_t ldd,
                        int32_t dim, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K8  weight gradients on tcgen05 (SURVEY 8f rank 4: the fine-tune step of a compacted expert,
 * pdm/training/trainer.py:1683-1765, differentiates F.conv2d / F.linear w.r.t. the weights).
 *   dw[n, tap, c] += sum_rows dy[row, n] * a[shift_tap(row), c]     (fp32, OHWI; taps = 9 if conv3x3 else 1)
 *   dbias[n]      += sum_rows dy[row, n]                            (optional)
 * dy: bf16 [rows, n_out] (pitch ld_dy), a: bf16 [rows, k_in] NHWC rows (pitch ld_a), rows = batch * H * W for the conv
 * (conv3x3 = 1: stride 1, zero padding 1; conv3x3 = 2: stride 2 -- H, W are the INPUT size, rows = batch * H/2 * W/2 and
 * k_in == ld_a); (bw, bh, bb) = box of OUTPUT pixels of one reduction stage (bw * bh * bb = 128, tiles the images);
 * splits = split-K factor over the rows (partial sums meet in dw through fp32 atomics: the caller zeroes dw / dbias).
 * ------------------------------------------------------------------------------------------------ */
int aptp_wgrad(const void* dy, int32_t ld_dy, const void* a, int32_t ld_a, float* dw, int64_t ld_dw, float* dbias,
               int64_t rows, int32_t n_out, int32_t k_in, int32_t conv3x3, int32_t batch, int32_t H, int32_t W,
               int32_t bw, int32_t bh, int32_t bb, int32_t splits, void* stream);
/* out[g, n] += sum of dy[row, n] over the rows_per_group consecutive rows of group g (fp32 [groups, n_out], row pitch out_ld, caller zeroes):
 * per-sample column sums = gradient of the time-embedding projection that is broadcast over a sample's pixels
 * (blocks.py:331-343). */
int aptp_col_sum_groups(const void* dy, int32_t ld, int32_t groups, int32_t rows_per_group, int32_t n_out, float* out,
                        int32_t out_ld, void* stream);

/* Weight-training variants of the norm backward (affine parameters trainable, as in the fine-tune stage):
 * aptp_groupnorm_bwd_affine = aptp_groupnorm_bwd that ALSO accumulates daffine[c] = (dgamma[c], dbeta[c]) (fp32 [C][2],
 * caller zeroes) in the same pass over x and da; aptp_layernorm_affine_bwd accumulates the same pair for LayerNorm
 * (dy = gradient of the LayerNorm output) in one extra pass with per-row statistics recomputed. */
int aptp_groupnorm_bwd_affine(const void* x, int32_t ldx, const void* da, int32_t ldda, void* dx, int32_t lddx,
                              int32_t accumulate, int32_t batch, int32_t hw, int32_t C, int32_t group_size, float eps,
                              const float* stats, int32_t stats_groups, const float* gamma, const float* beta,
                              const float* gate, int32_t gate_ld, int32_t silu, float* bstats, float* dgate,
                              float* daffine, void* stream);
int aptp_layernorm_affine_bwd(const void* x, int32_t ldx, const void* dy, int32_t lddy, int64_t rows, int32_t C, float eps,
                              float* daffine, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K9  small fp32 operators of the pruning train step (no cuBLAS / eager PyTorch left on the path).
 * ---------------------------------------------------------------------------------------------- */
/* HyperStructure._forward (pdm/models/hypernet/hypernet.py:72-79) over the row-concatenated 71 Linears:
 * y[B,N] = x[B,K] w[N,K]^T + bias[N]; backward: dw[N,K], db[N] (NULL to skip), dx[B,K] (NULL to skip). fp32 SIMT,
 * fixed summation order (the logits feed the router, whose assignments must be reproducible). */
int aptp_linear_f32_fwd(const float* x, const float* w, const float* bias, float* y, int32_t B, int32_t K, int32_t N,
                        void* stream);
int aptp_linear_f32_bwd(const float* x, const float* w, const float* dy, float* dx, float* dw, float* db, int32_t B,
                        int32_t K, int32_t N, void* stream);
/* ContrastiveLoss.forward (pdm/losses/contrastive_loss.py:11-22) over the all-gathered batch of M rows:
 * loss = BCE(softmax(A A^T / arch_temp)^T, softmax(P P^T / prompt_temp)^T), A / P = row-normalised arch / prompt rows.
 * Workspaces (device, fp32): inv_a[M], inv_p[M], Sa[M*M], Sp[M*M] (kept for the backward), row_loss[M]; loss[1].
 * Backward: darch[M,Da] = d loss / d arch * grad_loss[0]; workspaces dG[M*M], dhat[M*Da]. */
int aptp_contrastive_fwd(const float* arch, int32_t Da, const float* prompt, int32_t Dp, int32_t M, float arch_temp,
                         float prompt_temp, float* inv_a, float* inv_p, float* Sa, float* Sp, float* row_loss, float* loss,
                         void* stream);
int aptp_contrastive_bwd(const float* arch, int32_t Da, int32_t M, float arch_temp, const float* inv_a, const float* Sa,
                         const float* Sp, const float* grad_loss, float* dG, float* dhat, float* darch, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* APTP_SM100_H */
