/*
 * motionclone_b200 — C ABI of the B200 (sm_100a) kernels behind MotionClone's guided denoising path.
 *
 * The reference (LPengYang/MotionClone) has no FFI: its "operator API" is a Python method surface executed by ATen /
 * cuBLAS / xformers kernels (SURVEY.md §8b). These entry points are what a binding for that surface calls; each one
 * cites the reference lines whose arithmetic it replaces (paths relative to /root/reference/motionclone/).
 *
 * Conventions (all entry points):
 *   - plain C types only: device pointers, sizes, ELEMENT strides, fp32 scalars, the CUDA stream as void*;
 *   - enqueue-only: no allocation, no synchronisation, no global state except the error string and a launch counter;
 *   - return 0 on success, a negative MC_E_* code otherwise (mc_last_error() has the text); the Python wrapper raises;
 *   - fp16 storage ("half" = IEEE binary16), fp32 accumulation; index tensors are uint8.
 *
 * Temporal layout. A temporal tensor X (q, k, v, o, gradients) holds element (b, f, p, c) — batch, frame, spatial
 * position, channel — at  X + b*stride_b + f*stride_f + p*stride_p + c  (channels contiguous, c = h*DH + e).
 * The reference's "(b f) d c -> (b d) f c" rearranges (models/motion_module.py:279, :343) and head splits
 * (models/attention.py:367-379) are therefore never materialised: they are strides.
 * Per-row outputs (probabilities, top-1, gathered probabilities) use the reference's own order
 * [(b d), heads, f(query), f(key)] (utils/motionclone_functions.py:280).
 */
#ifndef MOTIONCLONE_B200_H_
#define MOTIONCLONE_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MC_ABI_VERSION 2

#define MC_OK 0
#define MC_E_INVALID (-1)     /* bad argument (null pointer, unsupported shape, misaligned stride) */
#define MC_E_UNSUPPORTED (-2) /* shape outside the compiled instantiations (L, head dim) */
#define MC_E_CUDA (-3)        /* launch failed; mc_last_error() carries cudaGetErrorString */

typedef struct mc_temporal_layout {
  int64_t stride_b, stride_f, stride_p; /* in elements; channel stride is 1 */
} mc_temporal_layout;

/* library identity / diagnostics */
int mc_abi_version(void);
const char* mc_last_error(void);
/* number of kernels this library has enqueued since load / since the last reset (bench.py "gpu_launches") */
uint64_t mc_launch_count(void);
void mc_reset_launch_count(void);
/* a CUDA-graph replay re-executes kernels this library enqueued during capture without passing through its entry points:
 * the host adds their number (the counter's delta over the capture) per replay */
void mc_add_launch_count(uint64_t n);

/*
 * Fused temporal self-attention forward: O = softmax(scale * Q K^T) V over the frame axis for every
 * (batch, position, head). Replaces VersatileAttention's core, models/motion_module.py:309-332 ->
 * models/attention.py:461-490 (baddbmm -> softmax -> bmm, scores and probabilities rounded to fp16 as there),
 * and optionally, from the same tile,
 *   probs      [B*D, H, L, L] fp16 : get_attention_scores, models/attention.py:564-611 (utils/motionclone_functions.py:279)
 *   top_val/top_idx [B*D, H, L]    : torch.topk(k=1) + uint8 cast, utils/motionclone_functions.py:79 (ties: lowest index)
 *   gathered   [B*D, H, L] fp16    : torch.gather(P, idx_ref), utils/motionclone_functions.py:91-92
 * Any of o, probs, top_val/top_idx, gather_idx/gathered may be NULL (v may be NULL iff o is NULL).
 * L in {8, 16, 32} (positional encoding max_len is 32, models/motion_module.py:60); DH in {8,16,32,40,64,80,128,160}.
 */
int mc_temporal_attn_fwd(const void* q, const void* k, const void* v, mc_temporal_layout qkv_layout,
                         void* o, mc_temporal_layout o_layout,
                         void* probs, void* top_val, uint8_t* top_idx,
                         const uint8_t* gather_idx, void* gathered,
                         int B, int D, int L, int H, int DH, float scale, void* stream);

/*
 * Backward of the above w.r.t. q, k, v (autograd of models/attention.py:461-490 plus the probability branch of
 * utils/motionclone_functions.py:260-283 that torch.autograd.grad traverses at :236). Probabilities are recomputed.
 * Incoming gradients, all optional (NULL):
 *   d_o        : gradient of O (layout do_layout)
 *   d_probs    : dense gradient of probs [B*D, H, L, L] fp16
 *   gather_idx + d_gathered [B*D, H, L] : one-hot gradient of the gathered probabilities (closed form of
 *                gather + mse_loss backward, utils/motionclone_functions.py:92-96)
 * Outputs dq, dk (and dv unless NULL) share g_layout.
 */
int mc_temporal_attn_bwd(const void* q, const void* k, const void* v, mc_temporal_layout qkv_layout,
                         const void* d_o, mc_temporal_layout do_layout,
                         const void* d_probs, const uint8_t* gather_idx, const void* d_gathered,
                         void* dq, void* dk, void* dv, mc_temporal_layout g_layout,
                         int B, int D, int L, int H, int DH, float scale, void* stream);

/* torch.topk(k=1, dim=-1) over fp16 rows of length L (utils/motionclone_functions.py:79); rows = product of the
 * leading dims. Stand-alone form of the fused epilogue above. */
int mc_top1_rows(const void* probs, int64_t rows, int L, void* top_val, uint8_t* top_idx, void* stream);

/*
 * Motion-guidance loss (utils/motionclone_functions.py:85-100) on gathered probabilities:
 *   loss_per_module[m] = fp16( mean_i fp16(fp16(cur_m[i] - ref_m[i])^2) ),  loss_total = fp16(sum_m loss_per_module[m])
 * (the rounding sequence of F.mse_loss on half tensors followed by stack().sum()). M <= 16 modules.
 */
int mc_motion_loss_fwd(int M, const void* const* cur, const void* const* ref, const int64_t* n,
                       void* loss_per_module, void* loss_total, void* stream);
/* d cur_m[i] = g * 2 (cur_m[i] - ref_m[i]) / n_m, with g read from device memory (fp16 scalar, no host sync). */
int mc_motion_loss_bwd(int M, const void* const* cur, const void* const* ref, const int64_t* n,
                       const void* d_loss_total, void* const* d_cur, void* stream);

/*
 * CFG combine + score-guided DDIM update in one pass (utils/motionclone_functions.py:239/:255 and :339-389, eta = 0,
 * epsilon prediction), replicating the eager fp16 rounding sequence op by op:
 *   d=h(ec-eu); m=h(cfg*d); e=h(ec+m); t1=h(sb*e); t2=h(x-t1); x0=h(t2*inv_sa);
 *   [g2=h(sc*score); e2=h(e-g2)] ; dir=h(c*e2); t3=h(sap*x0); x_prev=h(t3+dir)
 * sb=sqrt(1-a_t), inv_sa=1/sqrt(a_t), sap=sqrt(a_prev), c=sqrt(1-a_prev), sc=guidance_scale*sqrt(1-a_t) (fp32).
 * score may be NULL (plain step); eps_uncond may be NULL (eps_cond then IS the combined eps, as in the reference's
 * customized_step(model_output, ...) signature). n = element count.
 */
int mc_cfg_ddim_step(const void* eps_cond, const void* eps_uncond, const void* x, const void* score, void* x_prev,
                     int64_t n, float cfg_scale, float sqrt_beta_t, float inv_sqrt_alpha_t, float sqrt_alpha_prev,
                     float dir_coef, float score_coef, void* stream);

/* add_noise, utils/motionclone_functions.py:19-23: out = h(h(sa*x0) + h(sb*noise)). */
int mc_add_noise(const void* x0, const void* noise, void* out, int64_t n, float sqrt_alpha, float sqrt_one_minus_alpha,
                 void* stream);

/*
 * Text cross-attention forward on tcgen05 tensor cores with TMEM accumulators (csrc/cross_attn_fwd_tc.cu):
 * O = softmax(scale * Q K^T) V per (batch, head), Q [B, Nq, H*DH] (all frames of one prompt), K, V [B, Nk <= 80, H*DH].
 * Replaces the xformers call for `attn2` (models/attention.py:193-201, :280-285 -> :535-542).
 * Strides in elements (multiples of 8); head h occupies columns [h*DH, (h+1)*DH).
 * DH in {8, 16, 32, 40, 64, 80, 160}.
 */
int mc_cross_attn_fwd(const void* q, const void* k, const void* v, void* o, int B, int Nq, int Nk, int H, int DH,
                      int64_t q_stride_b, int64_t q_stride_row, int64_t kv_stride_b, int64_t kv_stride_row,
                      int64_t o_stride_b, int64_t o_stride_row, float scale, void* stream);

/*
 * Gradient of the same cross-attention with respect to Q only (tcgen05, csrc/cross_attn_bwd_tc.cu):
 * dQ = scale * [P o (dO V^T - rowsum(P o dO V^T))] K with P recomputed from Q, K. The text K / V are projections of a
 * constant prompt embedding through frozen weights (t2v_video_sample.py:67-68), so torch.autograd.grad w.r.t. the
 * latents (utils/motionclone_functions.py:236) never asks for dK / dV; the Python wrapper raises if it is asked to.
 * Same shape / stride rules as mc_cross_attn_fwd; d_o and dq are [B, Nq, H*DH] with their own strides.
 */
int mc_cross_attn_bwd_dq(const void* q, const void* k, const void* v, const void* d_o, void* dq, int B, int Nq, int Nk,
                         int H, int DH, int64_t q_stride_b, int64_t q_stride_row, int64_t kv_stride_b,
                         int64_t kv_stride_row, int64_t do_stride_b, int64_t do_stride_row, int64_t dq_stride_b,
                         int64_t dq_stride_row, float scale, void* stream);

/*
 * Spatial self-attention on tcgen05 tensor cores with TMEM accumulators and tensor-map TMA operand loads
 * (csrc/spatial_attn_tc.cu): O = softmax(scale * Q K^T) V per (frame, head) over the N tokens of one frame, any N >= 1
 * (128-key tiles, online softmax). Replaces the xformers call for `attn1`
 * (models/attention.py:190-192, :271-278 -> :535-542, xformers.ops.memory_efficient_attention, attn_bias=None).
 * q, k, v, o: [B, N, H*DH] views with their own frame / token strides in elements (multiples of 8; 16-byte aligned
 * pointers), head h in columns [h*DH, (h+1)*DH) - e.g. the column blocks of one fused QKV projection.
 * lse (nullable): fp32 [B, H, N], natural-log sum-exp of the scaled scores, kept for the backward.
 * DH in {8, 16, 32, 40, 64, 80, 160}.
 */
int mc_spatial_attn_fwd(const void* q, const void* k, const void* v, void* o, float* lse, int B, int N, int H, int DH,
                        int64_t q_stride_b, int64_t q_stride_row, int64_t k_stride_b, int64_t k_stride_row,
                        int64_t v_stride_b, int64_t v_stride_row, int64_t o_stride_b, int64_t o_stride_row, float scale,
                        void* stream);

/*
 * Backward of mc_spatial_attn_fwd w.r.t. q, k, v (the autograd of the xformers seam that torch.autograd.grad traverses,
 * utils/motionclone_functions.py:236): dV = P^T dO, dS = scale * P o (dO V^T - rowsum(dO o O)), dQ = dS K, dK = dS^T Q,
 * with P recomputed from the forward's log-sum-exp `lse` [B, H, N]. Three launches: rowsum(dO o O) -> workspace, a dQ
 * kernel (128-query CTAs streaming 64-key tiles) and a dK/dV kernel (128-key CTAs streaming 64-query tiles); tcgen05 +
 * TMEM + tensor-map TMA throughout, no atomics (deterministic). o, d_o: [B, N, H*DH] with their own strides; dq, dk, dv
 * share g_stride_* (e.g. the column blocks of one fused [B, N, 3*H*DH] gradient buffer).
 * workspace: mc_spatial_attn_bwd_workspace_bytes(B, N, H) bytes of device memory (fp32 [B, H, N]).
 */
int64_t mc_spatial_attn_bwd_workspace_bytes(int B, int N, int H);
int mc_spatial_attn_bwd(const void* q, const void* k, const void* v, const void* o, const void* d_o, const float* lse,
                        void* dq, void* dk, void* dv, void* workspace, int B, int N, int H, int DH, int64_t q_stride_b,
                        int64_t q_stride_row, int64_t k_stride_b, int64_t k_stride_row, int64_t v_stride_b,
                        int64_t v_stride_row, int64_t o_stride_b, int64_t o_stride_row, int64_t do_stride_b,
                        int64_t do_stride_row, int64_t g_stride_b, int64_t g_stride_row, float scale, void* stream);

/* out = a + bias[c] + b on channel-innermost fp16 tensors (n elements, C channels): the resnet's residual add
 * `input_tensor + hidden_states` (models/resnet.py:209-211) with conv2's (+ the shortcut conv's) bias folded in. */
int mc_bias_residual_add(const void* a, const void* b, const void* bias, void* out, int64_t n, int C, void* stream);

/*
 * Memory-bound glue of the UNet3D forward (and of the guided pass's backward) on NHWC / token-major fp16 activations.
 *
 * GroupNorm over channels_last x [N, HW, C] (N = batch*frames, N <= 1024) with G groups, optional fused SiLU
 * (csrc/groupnorm.cu): replaces InflatedGroupNorm + nonlinearity (models/resnet.py:21-29, :186-187, :197-204) and the
 * transformer input norms (models/attention.py:61,105; models/motion_module.py:112,145). Two launches: partial
 * (count, mean, M2) per split, folded into (mean, rstd) by the last CTA of each frame, then apply.
 * workspace: >= mc_groupnorm_workspace_bytes(N, G) bytes of device memory whose FIRST 4096 BYTES ARE ZERO on first use
 * (per-frame tickets; every call leaves them zero). One workspace per concurrently running stream.
 */
int64_t mc_groupnorm_workspace_bytes(int N, int G);
/* chan_bias (nullable): fp16 [N / frames_per_bias_row, C] added to x before the statistics and the normalisation —
 * the resnet's time-embedding add `hidden_states + temb` (models/resnet.py:194-195) folded into the norm that follows. */
int mc_groupnorm_nhwc(const void* x, const void* chan_bias, int frames_per_bias_row, void* y, const void* gamma,
                      const void* beta, void* workspace, int64_t workspace_bytes, int N, int HW, int C, int G, float eps,
                      int fuse_silu, void* stream);
/* LayerNorm over the last dim (models/attention.py:189,206,212; models/motion_module.py:204,210), C % 8 == 0, C <= 2048.
 * post_add (nullable): fp16 [frames, C] added after the norm to row r at frame (r / rows_per_frame) % frames - the
 * temporal positional encoding `x + pe[:, :f]` (models/motion_module.py:246, :281-282) on (b f)-major tokens.
 * pre_bias (nullable): fp16 [C] added to x before the statistics (LayerNorm(x + pre_bias)). Used by the transformer
 * blocks to carry the constant output biases of their projections inside the residual stream, so that every
 * `residual + Linear(x)` of a block is ONE GEMM with beta = 1 instead of a GEMM and an elementwise pass
 * (models/attention.py:271-300, models/motion_module.py:213-225). */
int mc_layernorm(const void* x, void* y, const void* gamma, const void* beta, const void* post_add, const void* pre_bias,
                 int rows_per_frame, int frames, int64_t rows, int C, float eps, void* stream);
/* Backward of the three (input gradients only: weights are frozen on this path, t2v_video_sample.py:67-68).
 * mc_groupnorm_nhwc_stats copies the forward's finalised statistics out of its workspace: stats [N, G, 2] = (mean, rstd)
 * fp32, kept for the backward. mc_groupnorm_nhwc_bwd needs its own workspace (same size and zero-ticket rule). */
int mc_groupnorm_nhwc_stats(const void* workspace, void* stats, int N, int HW, int G, float eps, void* stream);
int mc_groupnorm_nhwc_bwd(const void* x, const void* chan_bias, int frames_per_bias_row, const void* dz, void* dx,
                          const void* stats, const void* gamma, const void* beta, void* workspace,
                          int64_t workspace_bytes, int N, int HW, int C, int G, int fuse_silu, void* stream);
int mc_layernorm_bwd(const void* x, const void* dy, void* dx, const void* gamma, const void* pre_bias, int64_t rows, int C,
                     float eps, void* stream);
int mc_geglu_bwd(const void* in, const void* dout, void* din, int64_t T, int I, void* stream);
/* GEGLU of diffusers-0.16 FeedForward (models/attention.py:211, models/motion_module.py:209):
 * in [T, 2I] = [h | gate] -> out [T, I] = h * gelu_erf(gate), gelu output rounded to fp16 as in the eager graph */
int mc_geglu(const void* in, void* out, int64_t T, int I, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MOTIONCLONE_B200_H_ */
