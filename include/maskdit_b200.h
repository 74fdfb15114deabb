/* maskdit_b200 — C ABI of the B200 (sm_100a) MaskDiT hot path.
 *
 * The reference (Anima-Lab/MaskDiT) is pure Python/PyTorch and has no FFI layer; its seam for this path is the
 * Python registries `Precond_models`, `DiT_models` (models/maskdit.py:709-715,779-781), `Losses`
 * (train_utils/loss.py:66-68) and `edm_sampler` (sample.py:30-66).  The Python shim in `maskdit_b200/` implements
 * those registries and calls the functions below through ctypes.  Every function:
 *   - takes raw DEVICE pointers + sizes + a `cudaStream_t` (passed as void*), no torch types;
 *   - is asynchronous on that stream, allocates nothing, frees nothing (caller owns all buffers);
 *   - returns MDT_OK (0) or a negative MDT_ERR_* code; the shim raises on non-zero.
 * Each declaration cites the reference code (file:line in /root/reference) whose arithmetic it replaces.
 */
#ifndef MASKDIT_B200_H_
#define MASKDIT_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MDT_OK 0
#define MDT_ERR_ARG (-1)    /* bad shape / alignment / null pointer */
#define MDT_ERR_CUDA (-2)   /* launch failed; see cudaGetLastError */
#define MDT_ERR_DRIVER (-3) /* cuTensorMapEncodeTiled entry point unavailable */
#define MDT_ERR_TMAP (-4)   /* tensor-map encode rejected the operand */
#define MDT_ERR_UNSUPPORTED (-5)

const char* mdt_status_string(int status);
int mdt_abi_version(void);
/* BLOCK_N * 10 + CTAs-per-tile (1 or 2 = tcgen05 cta_group::2 SM pair) of the last mdt_gemm_bf16 launch (tests). */
int mdt_gemm_last_config(void);
/* Bit set of the GEMM instances launched since the last reset: bit (BLOCK_N/64 - 2) * 2 + (CTAs - 1), i.e. 128/1 = 0,
 * 128/2 = 1, 192/1 = 2, 192/2 = 3, 256/1 = 4, 256/2 = 5.  reset != 0 clears it after reading.                        */
int mdt_gemm_configs_seen(int reset);

/* ------------------------------------------------------------------------------------------------------------
 * bf16 tensor-core GEMM (tcgen05 / TMEM / TMA):  out[M,N] (+)= sum_k A[m,k] * B[n,k], fp32 accumulate.
 * Replaces every nn.Linear forward and its autograd dgrad/wgrad: timm Attention.qkv/proj and Mlp.fc1/fc2
 * (ctor sites models/maskdit.py:178,182), adaLN_modulation (:185,206,227), DecoderLayer.linear (:203),
 * FinalLayer.linear (:224), TimestepEmbedder.mlp (:34-38), LabelEmbedder.embedding_table (:75).
 *   a_mn / b_mn = 0: operand stored [rows, K] with K contiguous ("K-major", row stride lda/ldb elements)
 *               = 1: operand stored [K, rows] with rows contiguous ("MN-major")
 * ------------------------------------------------------------------------------------------------------------ */
enum { MDT_EPI_STORE = 0,      /* out = act(acc + bias [+ resid])            out bf16 or fp32            */
       MDT_EPI_GELU = 1,       /* aux = bf16(acc+bias); out = bf16(gelu_tanh(aux))      (Mlp.fc1 + act)   */
       MDT_EPI_GATE_RESID = 2, /* y = acc+bias; aux = bf16(y) (optional); out_f32 = resid + gate[row/rpg]*y
                                  (DiTBlock residual update, models/maskdit.py:190-191)                   */
       MDT_EPI_DGELU = 3,      /* out = bf16(acc * gelu_tanh'(aux))          (backward through GELU)      */
       MDT_EPI_ATOMIC = 4 };   /* out_f32 += acc via red.global.add, stream-K schedule (wgrad, long-K)    */
enum { MDT_ACT_NONE = 0, MDT_ACT_SILU = 1 };

typedef struct mdt_gemm_args {
  const void* A; /* bf16 */
  const void* B; /* bf16 */
  int M, N, K;
  int lda, ldb;  /* row strides in elements (multiple of 8) */
  int a_mn, b_mn;
  int epi, act;
  void* out;
  int ldo;       /* multiple of 8 */
  int out_fp32;  /* 1: float output, 0: bf16 output */
  const float* bias; /* [N] or NULL */
  void* aux;     /* bf16 [M, ld_aux], see epilogue kinds */
  int ld_aux;
  const float* resid; /* fp32 [M, ld_resid] or NULL */
  int ld_resid;
  const float* gate;  /* fp32 [M / rows_per_group, ld_gate] */
  int ld_gate;
  int rows_per_group;
  int block_n;   /* 0 = auto, or 128/192/256 */
  float* colsum; /* MDT_EPI_DGELU only, may be NULL: colsum[n] += sum_m out[m,n] (the bf16-rounded outputs), i.e. the
                    bias gradient of the layer whose pre-activation gradient this GEMM produces (fp32 red.add)      */
} mdt_gemm_args;

int mdt_gemm_bf16(const mdt_gemm_args* args, void* stream);
/* The host-side decisions mdt_gemm_bf16 would take for `args`, without launching anything (needs no device: host
 * tests pin the dispatch with it; pointers in `args` are only checked for alignment, never dereferenced):
 * out10 = {BLOCK_N, CTAs per tile (2 = cta_group::2 SM pair), k-slices, paired half-tile order (0/1), half-width last
 * column tile (0/1), row tiles, column tiles, k-blocks of 64, work units, grid size in CTAs}.                        */
int mdt_gemm_plan(const mdt_gemm_args* args, long long* out10);
/* Measurement aid (bench.py roofline): while enabled, every mdt_gemm_bf16 launch of this process - also the step
 * driver's - is bracketed by CUDA events on its stream; mdt_gemm_profile_read returns the launch count and fills
 * ms[i] (device time) / flops[i] (2 M N K) for i < cap.  Enabling clears the previous recording.                   */
int mdt_gemm_profile_enable(int on);
int mdt_gemm_profile_read(float* ms, double* flops, int cap);

/* ------------------------------------------------------------------------------------------------------------
 * Mask index path (integer, bit-exact).  get_mask, models/maskdit.py:88-113: ids_shuffle = argsort(noise),
 * ids_restore = argsort(ids_shuffle), ids_keep = ids_shuffle[:, :len_keep], mask = (ids_restore >= len_keep).
 * Ties in `noise` are broken by ascending index (= torch.argsort(stable=True)).
 *   noise [B,L] f32 -> ids_keep [B,len_keep] i64, ids_restore [B,L] i64, mask [B,L] f32 (0 keep / 1 remove)
 * ------------------------------------------------------------------------------------------------------------ */
int mdt_mask_indices(const float* noise, int B, int L, int len_keep, int64_t* ids_keep, int64_t* ids_restore,
                     float* mask, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * PatchEmbed + pos_embed + mask_out_token + EDM c_in scaling, fused.
 * models/maskdit.py:475 (x_embedder(x) + pos_embed), :126 (gather kept tokens), :764-769 (c_in * x).
 *   x [B,C,R,R] f32, sigma [B] f32 or NULL (c_in = 1/sqrt(sigma_data^2+sigma^2), 1 if NULL),
 *   W [D, C*p*p] f32 (Conv2d weight flattened (c,ph,pw)), bias [D], pos [L,D] f32,
 *   ids_keep [B,T] i64 or NULL (NULL: T == L, identity) -> out [B,T,D] f32
 * Backward: gW [D, C*p*p] += sum g (x) patch, gb [D] += sum g    (no input gradient is needed)
 * ------------------------------------------------------------------------------------------------------------ */
int mdt_patch_embed(const float* x, const float* sigma, float sigma_data, const float* W, const float* bias,
                    const float* pos, const int64_t* ids_keep, float* out, int B, int C, int R, int p, int D, int T,
                    void* stream);
int mdt_patch_embed_bwd(const float* x, const float* sigma, float sigma_data, const int64_t* ids_keep,
                        const float* g, float* gW, float* gb, int B, int C, int R, int p, int D, int T, void* stream);

/* TimestepEmbedder.timestep_embedding (models/maskdit.py:41-58) on t = c_noise = ln(sigma)/4 (:767):
 *   out[b] = [cos(t f_k) | sin(t f_k)], f_k = exp(-ln(1e4) k / (dim/2)); out bf16 [B, dim]                  */
int mdt_timestep_freq(const float* sigma, int B, int dim, void* out_bf16, void* stream);

/* Pointwise helpers around the conditioning MLPs (nn.SiLU at models/maskdit.py:36,184,205,226).
 *   silu:      out_bf16 = silu(a [+ b])  (and out_f32 = a + b if non-NULL)
 *   silu_bwd:  dx = dy * silu'(x)                                                                            */
int mdt_silu(const float* a, const float* b, float* sum_f32, void* out_bf16, long long n, void* stream);
int mdt_silu_bwd(const float* dy, const float* x, float* dx_f32, void* dx_bf16, long long n, void* stream);
int mdt_cast_f32_bf16(const float* in, void* out_bf16, long long n, void* stream);
/* column sums: out[N] (+)= sum_m in[m, n]  (bias gradients) */
int mdt_colsum_bf16(const void* in_bf16, int M, int N, int ld, float* out, void* stream);
int mdt_colsum_f32(const float* in, int M, int N, int ld, float* out, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * LayerNorm(no affine, eps) + modulate, models/maskdit.py:19-20,177,179,190-191,202,211,223,232:
 *   out_bf16[m,:] = LN(x[m,:]) * (1 + scale[m / rows_per_group,:]) + shift[m / rows_per_group,:]
 * saves mean/rstd [M] for the backward.  shift/scale are fp32 with row stride ld_mod.
 * Backward (dxmod bf16 -> residual-stream gradient, fp32):
 *   g[m,:] (+)= d LN / dx ; dshift[b,:] += sum_t dxmod ; dscale[b,:] += sum_t dxmod * xhat
 * ------------------------------------------------------------------------------------------------------------ */
int mdt_ln_modulate(const float* x, const float* shift, const float* scale, int ld_mod, int rows_per_group,
                    void* out_bf16, float* mean, float* rstd, int M, int D, float eps, void* stream);
int mdt_ln_modulate_bwd(const void* dxmod_bf16, const float* x, const float* mean, const float* rstd,
                        const float* scale, int ld_mod, int rows_per_group, float* g, int accumulate,
                        float* dshift, float* dscale, int ld_dmod, int M, int D, void* stream);

/* Backward of  x_out = x + gate * y  (models/maskdit.py:190-191) w.r.t. y and gate, plus the bias gradient of the
 * Linear that produced y:  dy_bf16 = g * gate ; dgate[b,:] += sum_t g*y ; dbias[:] += sum_m dy                 */
int mdt_gate_bwd(const float* g, const void* y_bf16, const float* gate, int ld_gate, int rows_per_group,
                 void* dy_bf16, float* dgate, int ld_dgate, float* dbias, int M, int D, void* stream);

/* mdt_ln_modulate_bwd immediately followed by mdt_gate_bwd on the finished residual gradient g, in one pass
 * (the block backward alternates exactly these two: models/maskdit.py:190-191 differentiated right to left).
 * y_bf16 == NULL: LN backward only.  Same arguments and arithmetic as the two separate entry points.          */
int mdt_ln_modulate_bwd_gate(const void* dxmod_bf16, const float* x, const float* mean, const float* rstd,
                             const float* scale, int ld_mod, int rows_per_group, float* g, int accumulate,
                             float* dshift, float* dscale, int ld_dmod, const void* y_bf16, const float* gate,
                             int ld_gate, void* dy_bf16, float* dgate, int ld_dgate, float* dbias, int M, int D,
                             void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Multi-head attention core of timm Attention (ctor models/maskdit.py:178):
 *   qkv [B,T,3,H,dh] bf16 -> out [B,T,H*dh] bf16 = softmax(q k^T / sqrt(dh)) v ; lse [B,H,T] f32 (log-sum-exp)
 * Backward: dqkv [B,T,3,H,dh] bf16 from dout.
 * ------------------------------------------------------------------------------------------------------------ */
int mdt_attention_fwd(const void* qkv, void* out, float* lse, int B, int T, int H, int dh, void* stream);
int mdt_attention_bwd(const void* qkv, const void* out, const void* dout, const float* lse, void* dqkv, int B, int T,
                      int H, int dh, void* stream);
/* Introspection for the parity tests (host-side, no launch): which kernel family served the last successful
 * mdt_attention_fwd (which = 0) / mdt_attention_bwd (which = 1) call of this process:
 *   0 mma.sync fallback (odd sequence lengths), 1 split-tile TMA tcgen05 (T = 128/256), 2 no-swizzle tcgen05,
 *   3 blocked split-tile tcgen05 (T = 512/1024, T = 256 backward), 4 blocked no-swizzle tcgen05; -1 = none yet.
 * With MDT_ATTN_STRICT=1 in the environment a shape no tcgen05 kernel accepts returns MDT_ERR_UNSUPPORTED instead
 * of running the mma.sync kernels.                                                                             */
int mdt_attention_last_impl(int which);
/* Log of every attention call since the last reset, 4 ints per call: (which, T, head_dim, kernel family).  Returns
 * the number of entries copied (<= cap); out4 == NULL resets the log.  The step driver's internal calls are logged too. */
int mdt_attention_impl_log(int* out4, int cap);

/* ------------------------------------------------------------------------------------------------------------
 * unmask_tokens + decoder_pos_embed (models/maskdit.py:157-163,543-545):
 *   out[b,l,:] = (ids_restore[b,l] < T ? u[b, ids_restore[b,l], :] : mask_token) + pos[l,:]
 * ids_restore NULL = eval path (no masking): out = u + pos.
 * Backward: du_bf16[b,i,:] = g[b, ids_keep[b,i], :] ; dmask_token[:] += sum over removed positions of g.
 * ------------------------------------------------------------------------------------------------------------ */
int mdt_unmask_tokens(const float* u, const float* mask_token, const float* pos, const int64_t* ids_restore,
                      float* out, int B, int T, int L, int D, void* stream);
int mdt_unmask_tokens_bwd(const float* g, const int64_t* ids_keep, const int64_t* ids_restore, void* du_bf16,
                          float* dmask_token, int B, int T, int L, int D, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * unpatchify + EDM preconditioning + EDM/MAE loss, forward and the gradient seed in one pass.
 *   F [B,L,p*p*C] f32 (final_layer output) ; xin [B,C,R,R] noisy input y+n ; y [B,C,R,R] clean ; sigma [B]
 *   D = c_skip*xin + c_out*unpatchify(F)                    models/maskdit.py:411-424,764-771
 *   mask != NULL: loss[b] = mean_{kept}(patch-mean(w (D-y)^2)) + mae_coef * mean_{removed}(MSE(patchify(D), norm-patchify(xin)))
 *                                                            train_utils/loss.py:37,44-52,73-101
 *   mask == NULL: loss[b] = mean(w (D-y)^2)                  loss.py:54
 *   dF_bf16 (optional) = d(sum_b gl[b]*loss[b]) / dF ; Dx (optional) [B,C,R,R] f32.
 * ------------------------------------------------------------------------------------------------------------ */
int mdt_edm_loss(const float* F, const float* xin, const float* y, const float* sigma, const float* mask,
                 const float* gl, float sigma_data, float mae_coef, float* loss, float* Dx, void* dF_bf16, int B,
                 int C, int R, int p, void* stream);
/* Step front (train.py:206,209 + train_utils/loss.py:35-39 + utils.py:59-65) in one pass, given pre-drawn randoms:
 *   y  = scale_factor * (mean + exp(0.5 * clamp(logvar, -30, 20)) * eps)   moments [B,2C,R,R] = (mean | logvar)
 *   sigma[b] = exp(P_std * rnd_normal[b] + P_mean) ;  yn = y + noise_unit * sigma[b]
 *   labels[b,:] = 0 where !(drop_u[b] >= drop_prob)   (labels / drop_u may be NULL: no label dropout)
 * eps, noise_unit, y, yn: [B,C,R,R] f32 ; rnd_normal, drop_u, sigma: [B] f32 ; labels [B,num_classes] f32 in place. */
int mdt_step_front(const float* moments, const float* eps, const float* rnd_normal, const float* noise_unit,
                   const float* drop_u, float drop_prob, float scale_factor, float P_mean, float P_std, float* y,
                   float* yn, float* sigma, float* labels, int B, int C, int R, int num_classes, void* stream);

/* D only (sampler / generic autograd path): Dx = c_skip*xin + c_out*unpatchify(F); and its backward
 * dF_bf16 = c_out * patchify(gD).                                                                            */
int mdt_edm_precond_out(const float* F, const float* xin, const float* sigma, float sigma_data, float* Dx, int B,
                        int C, int R, int p, void* stream);
int mdt_edm_precond_out_bwd(const float* gD, const float* sigma, float sigma_data, void* dF_bf16, int B, int C, int R,
                            int p, void* stream);

/* Classifier-free guidance combine (forward_with_cfg, models/maskdit.py:580-583) fused with the EDM output scaling:
 *   F [2B,L,p*p*C] (cond rows first, uncond rows second) -> Dx [B,C,R,R] = c_skip*x + c_out*(Fu + s (Fc - Fu))  */
int mdt_cfg_precond_out(const float* F, const float* xin, const float* sigma, float sigma_data, float cfg_scale,
                        float* Dx, int B, int C, int R, int p, void* stream);

/* EDM Heun sampler state update in fp64 (sample.py:56-64):
 *   mode 0 (Euler):  d_cur = (x_hat - den)/t_hat ; x_next = x_hat + (t_next - t_hat) d_cur
 *   mode 1 (Heun):   d_prime = (x_next - den)/t_next ; x_next = x_hat + (t_next - t_hat)(0.5 d_cur + 0.5 d_prime) */
int mdt_heun_update(int mode, const double* x_hat, const float* denoised, double* d_cur, double* x_next,
                    float* x_next_f32, double t_hat, double t_next, long long n, void* stream);

/* Generalised fp64 sampler update for ablation_sampler (sample.py:73-188; Euler / Heun / churn steps of every
 * discretization, schedule and scaling are linear combinations with host-computed fp64 scalars):
 *   out = a*x + b*y + c*z (x, y fp64; z fp32 network output; y / z may be NULL) ; out_f32 = float(out * f32_scale)
 *   (out or out_f32 may be NULL).                                                                                */
int mdt_lincomb_f64(double a, const double* x, double b, const double* y, double c, const float* z, double* out,
                    float* out_f32, double f32_scale, long long n, void* stream);

/* Sampler tail (sample.py:287): img [B,C,H,W] f32 in [-1,1] -> uint8 [B,H,W,C] = clamp((img + 1) * 127.5, 0, 255).  */
int mdt_to_uint8_nhwc(const float* img, unsigned char* out, int B, int C, int H, int W, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Fused AdamW (weight_decay handled as adam_w_mode, train.py:141) + EMA (train_utils/helper.py:47-58) + bf16
 * weight-shadow refresh over flat buffers:  one pass instead of apex multi_tensor_adam + a 376-launch EMA loop.
 *   g is multiplied by grad_scale first (1/world_size after a SUM all-reduce).  ema / w_bf16 may be NULL.
 *   max_blocks > 0 caps the grid (a background launch overlapped with the backward GEMMs needs only a few CTAs).
 * ------------------------------------------------------------------------------------------------------------ */
int mdt_adamw_ema(float* w, const float* g, float* m, float* v, float* ema, void* w_bf16, long long n, float lr,
                  float beta1, float beta2, float eps, float weight_decay, int step, float ema_decay,
                  float grad_scale, int max_blocks, void* stream);
/* Same with a bf16 gradient operand: the buffer a bf16 gradient all-reduce produced (SURVEY 8e: 1.46 GB instead of
 * 2.92 GB on the wire, fp32 moments / master weights unchanged).                                                  */
int mdt_adamw_ema_g16(float* w, const void* g_bf16, float* m, float* v, float* ema, void* w_bf16, long long n,
                      float lr, float beta1, float beta2, float eps, float weight_decay, int step, float ema_decay,
                      float grad_scale, int max_blocks, void* stream);

/* Cap on the SMs the persistent kernels (tcgen05 GEMM, persistent attention backward) occupy: n > 0 sizes their grids
 * for n SMs instead of the device's count, leaving the rest to a concurrently running collective (the gradient
 * all-reduce overlapped with the backward); 0 = whole device.  Host-side setting, read at launch.                  */
int mdt_set_sm_budget(int n);
int mdt_get_sm_budget(void);

/* ============================================================================================================
 * Step driver (SURVEY 8b): the whole network forward / backward as ONE call each over a packed parameter blob and ONE
 * caller-provided workspace — the launch sequence the reference obtains from autograd + torch.compile for
 * `loss = loss_fn(net, ...); loss.mean().backward()` (train.py:179,216-220; DiT.forward models/maskdit.py:467-557).
 * No allocation, no host synchronisation, everything enqueued on `stream`.
 *
 * Packed blob (element offsets shared by the fp32 master w32, the bf16 shadow w16 and the fp32 gradient):
 *   [adaLN_modulation.1.weight of blocks 0..depth-1, decoder_layer, decoder_blocks 0.., final_layer]
 *   [the matching adaLN biases] [all other trainable tensors in registration order] [pos_embed, decoder_pos_embed]
 * every tensor on a 64-element boundary; names = the reference's state-dict keys (models/maskdit.py:242-332).
 * ============================================================================================================ */
typedef struct mdt_model_cfg {
  int img_resolution, img_channels, patch_size, num_classes; /* EDMPrecond / DiT ctor, models/maskdit.py:722-741     */
  int hidden, depth, heads, mlp_hidden;                      /* encoder DiTBlocks (DiT_models, :645-715)              */
  int dec_hidden, dec_depth, dec_heads, dec_mlp_hidden;      /* decoder (:310-312: 512, 8, 16, 2048)                  */
  int has_mask_token;                                        /* mae_loss_coef > 0 (:297-299)                          */
  float sigma_data;
} mdt_model_cfg;
typedef struct mdt_model mdt_model; /* host-side layout object: no device memory, no CUDA calls */

int mdt_model_create(const mdt_model_cfg* cfg, mdt_model** out);
void mdt_model_destroy(mdt_model* m);
long long mdt_model_param_count(const mdt_model* m, int trainable_only); /* blob length in elements                  */
int mdt_model_num_tensors(const mdt_model* m);
/* i-th tensor in BLOB order: state-dict key, element offset, element count                                            */
int mdt_model_param_info(const mdt_model* m, int i, char* name, int name_cap, long long* offset, long long* numel);
int mdt_model_mod_width(const mdt_model* m); /* columns of the concatenated adaLN modulation vector                   */

/* Workspace bytes for batch B with T kept tokens per sample (T <= 0: no token dropping, T = L).
 * training != 0: every activation the backward needs stays resident (+ the backward's scratch); else inference.       */
long long mdt_workspace_bytes(const mdt_model* m, int B, int T, int training);

/* F [B*L, p*p*C] f32 = DiT.forward on x_in [B,C,R,R] (UNscaled network input, c_in applied inside), sigma [B],
 * labels [B,num_classes] f32 (NULL iff num_classes == 0), ids_keep [B,T] / ids_restore [B,L] int64 (both NULL: all
 * tokens).  save != 0 keeps the activations in `workspace` (256-byte aligned) for mdt_backward.                        */
int mdt_forward(const mdt_model* m, const float* w32, const void* w16, const float* x_in, const float* sigma,
                const float* labels, const int64_t* ids_keep, const int64_t* ids_restore, int B, int T, int save,
                void* workspace, long long workspace_bytes, float* F_out, void* stream);

/* grad (flat f32, blob offsets, trainable region) += d(loss)/d(params) given dF [B*L, p*p*C] bf16 and the workspace
 * of the matching mdt_forward(save = 1).  `on_ready(user, lo, hi)` (may be NULL) is called on the host as soon as the
 * kernels that finalise the gradient elements [lo, hi) of one block have been enqueued (DDP-bucket-style overlap).     */
typedef void (*mdt_grad_ready_fn)(void* user, long long lo, long long hi);
int mdt_backward(const mdt_model* m, const float* w32, const void* w16, float* grad, const float* x_in,
                 const float* sigma, const int64_t* ids_keep, const int64_t* ids_restore, const void* dF_bf16, int B,
                 int T, void* workspace, long long workspace_bytes, mdt_grad_ready_fn on_ready, void* user,
                 void* stream);

/* Data-parallel gradient exchange (train.py:178 DDP -> SURVEY 8e: ONE sum-all-reduce of the flat gradient buffer over
 * NVLink).  NCCL is resolved at run time from the process's libnccl.so.2 (MDT_ERR_DRIVER when absent).
 *   mdt_nccl_unique_id: rank 0 fills 128 bytes, the host code ships them to every rank (any side channel);
 *   mdt_nccl_comm_create: ncclCommInitRank (max_ctas > 0: ncclCommInitRankConfig with maxCTAs, a communicator that
 *   shares the GPU with the backward, see mdt_set_sm_budget); mdt_allreduce_grads: in-place SUM of fp32 (bf16 = 0) or
 *   bf16 elements.                                                                                                  */
int mdt_nccl_unique_id(void* id128);
int mdt_nccl_comm_create(const void* id128, int rank, int world, int max_ctas, void** comm);
int mdt_nccl_comm_destroy(void* comm);
int mdt_allreduce_grads(void* comm, void* grad, long long n, int bf16, void* stream);

/* ============================================================================================================
 * SD-VAE: decode, the sampler tail (sample.py:275 `vae.decode(z)`; autoencoder.py:306-453), and encode_moments, the
 * latent extraction in front of training (extract_latent.py:77; autoencoder.py:212-303,431-434).  Activations are
 * pixel-major fp32 row matrices [B*H*W, C]; every convolution is mdt_gemm_bf16 on an im2col operand built by
 * mdt_vae_im2col (GroupNorm(32) affine, swish and nearest-2x upsample of its source fused in) or mdt_vae_im2col_down.
 * The host sequencing is maskdit_b200/vae.py (same state-dict keys as FrozenAutoencoderKL).
 * ============================================================================================================ */
/* out [B*P, C] f32 = post_quant_conv(z / scale_factor), z [B,C,h,w] NCHW (autoencoder.py:449-451); C <= 8           */
int mdt_vae_post_quant(const float* z, const float* W, const float* bias, float scale_factor, float* out, int B,
                       int C, int P, void* stream);
/* GroupNorm(32) statistics (Normalize, autoencoder.py:34-35) of x [B,P,C] f32: sums [B,32,2] f64 = (sum, sum of squares),
 * deterministic (fixed-order two-pass reduction); scratch: B * ceil(P/256) * 64 floats                              */
int mdt_vae_gn_stats(const float* x, double* sums, float* scratch, int B, int P, int C, void* stream);
/* A [B*H*W, Kp] bf16, A[(b,y,x),(ky,kx,c)] = f(src[b,(y+ky-pad)/up,(x+kx-pad)/up,c]) (0 outside); ks = 1 | 3; up = 1 | 2;
 * f = identity (sums NULL) | GroupNorm affine | GroupNorm affine + swish (silu != 0): ResnetBlock / Upsample /
 * norm_out inputs (autoencoder.py:49-53,117-137,404-406); columns >= ks*ks*C are zero.                              */
int mdt_vae_im2col(const float* src, const double* sums, const float* gamma, const float* beta, int silu, int ks,
                   int up, void* A_bf16, int B, int H, int W, int C, int Kp, void* stream);
/* A [B*(H/2)*(W/2), Kp] bf16, A[(b,y,x),(ky,kx,c)] = src[b,2y+ky,2x+kx,c], 0 where 2y+ky >= H or 2x+kx >= W: the
 * F.pad(x,(0,1,0,1)) + 3x3 stride-2 convolution of Downsample (autoencoder.py:56-75).  src [B,H,W,C] f32 (H, W: source
 * dims, even); columns >= 9*C are zero.                                                                              */
int mdt_vae_im2col_down(const float* src, void* A_bf16, int B, int H, int W, int C, int Kp, void* stream);
/* x [B,3,H,W] f32 NCHW -> out [B*H*W, 4] f32 pixel-major rows, channel 3 = 0 (the encoder's conv_in input);
 * flip != 0 mirrors x along W (`img.flip(dims=[-1])`, extract_latent.py:85)                                          */
int mdt_vae_image_to_rows(const float* x, float* out, int B, int H, int W, int flip, void* stream);
/* moments [B,C,P] f32 NCHW = quant_conv(rows) (1x1, autoencoder.py:431-434), rows [B*P, ldx] f32 (first C columns); C <= 8 */
int mdt_vae_quant_out(const float* rows, int ldx, const float* W, const float* bias, float* moments, int B, int C,
                      int P, void* stream);
/* P [rows, cols] bf16 = softmax(scale * S) along columns (AttnBlock, autoencoder.py:185-187)                        */
int mdt_vae_softmax_rows(const float* S, float scale, void* P_bf16, int rows, int cols, void* stream);
/* the same with row stride ld >= cols for S and P; P[:, cols:ld] = 0 (T = h*w not a multiple of 8: the GEMMs need
 * 16-byte row strides)                                                                                                */
int mdt_vae_softmax_rows_ld(const float* S, float scale, void* P_bf16, int rows, int cols, int ld, void* stream);
/* x [B,P,ldx] f32 (first C columns) -> out [B,C,P] f32: the NCHW image `decode` returns                             */
int mdt_vae_rows_to_nchw(const float* x, float* out, int B, int P, int C, int ldx, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MASKDIT_B200_H_ */
