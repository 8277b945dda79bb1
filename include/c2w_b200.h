/* c2w_b200 — C ABI of the B200-native guided-sampling hot path of Climate2Weather.
 *
 * The reference (schmidtjonathan/Climate2Weather) has NO plugin / operator / FFI interface: its hot path is
 * three Python classes calling PyTorch library ops (SURVEY.md §8(b)).  Each entry point below therefore cites
 * the reference *function* (file:line under the reference root) whose arithmetic it replaces; the Python
 * mirror of those classes in climate2weather_b200/ is the only caller (ctypes, see INTEGRATION.md).
 *
 * Conventions: plain C, `int` return (0 = ok, negative = error, text via c2w_last_error()); the caller owns every
 * tensor and passes raw DEVICE pointers plus a cudaStream_t (as void*); the library owns only its handle, the
 * packed weights and the tensor maps it builds over the caller's workspace.  No hidden allocation and no
 * synchronisation on the hot calls.  One handle per device/process, not re-entrant per handle.
 *
 * Device layouts
 *   trajectory / score / noise : fp32 [frames, H, W, C]   (C = 4 variables -> one float4 per pixel)
 *   reference-facing tensors   : fp32 NCHW, converted by c2w_traj_pack / c2w_traj_unpack
 *   activations (internal)     : bf16 NHWC, channel counts padded to multiples of 64
 */
#ifndef C2W_B200_H
#define C2W_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define C2W_MAX_LEVELS 8

/* Architecture of model.score.ScoreUNet (model/score.py:37-57, model/nn.py:108-218, configs/sda_unet.yml). */
typedef struct c2w_config {
  int32_t frame_channels;                  /* C: variables per frame (train.py:169: channels = C * window) */
  int32_t window;                          /* w = 2k+1 frames per Markov window (run_training.sh:41)       */
  int32_t height, width;                   /* patch size (run_training.sh:39)                               */
  int32_t embedding_dim;                   /* configs/sda_unet.yml:1                                        */
  int32_t noise_features;                  /* model/score.py:53 (32)                                        */
  int32_t n_levels;
  int32_t hidden_channels[C2W_MAX_LEVELS]; /* configs/sda_unet.yml:8-13                                     */
  int32_t hidden_blocks[C2W_MAX_LEVELS];   /* configs/sda_unet.yml:2-7                                      */
  int32_t attention_mask;                  /* bit l set: AttentionBlock after every block of level l        */
  int32_t forcing_dim;                     /* model/score.py:46-51: Linear(forcing_dim, embedding_dim); 0 = none */
} c2w_config;

typedef struct c2w_handle c2w_handle;

/* Guided predictor / corrector arithmetic on the resident trajectory.
 * Replaces AbstractScoreFunction.condition_on/log_p + __call__ (src/thor/score.py:24-60, exact_grad=False closed
 * form), the observation operator A and its adjoint (exp/downscaling.py:129-132) and SDAPipeline._sample_step
 * (src/thor/pipelines.py:41-46) / the corrector body (src/thor/pipelines.py:81-88). */
#define C2W_MAX_VARS 8
typedef struct c2w_guide {
  float* x;             /* [frames_local, H, W, C] state, updated in place (mode 0)                       */
  const float* eps;     /* [frames_local, H, W, C] window-composed score                                   */
  float* eps_out;       /* mode 1: guided score                                                            */
  const float* y;       /* [ceil(L / t_step), C, H / s_step, W / s_step] observation; NULL = unconditioned */
  float std2[C2W_MAX_VARS]; /* likelihood std^2 per variable (exp/downscaling.py:221-227)                  */
  float gamma[C2W_MAX_VARS];
  float mu, sigma;           /* schedule at the score's time (src/thor/pipelines.py:13-20)                 */
  float mu_next, sigma_next; /* schedule at t - dt                                                         */
  int32_t t_step, s_step, H, W;
  int32_t frame_global0; /* global frame index of local frame 0 (time sharding)                            */
  int32_t own_lo, own_n; /* local frames [own_lo, own_lo + own_n) are updated                              */
  int32_t mode;          /* 0 predictor update, 1 guided eps + per-CTA partial sums of eps^2,
                            2 likelihood cotangent g = A^T((y - A x0)/var) -> cot_out (exact_grad)          */
  float* partials;       /* mode 1: >= own_n * (H / s_step) floats                                         */
  int32_t* nan_flag;     /* set to 1 if any updated value is not finite (src/thor/pipelines.py:90-91)      */
  const float* vjp;      /* exact_grad=True: J_eps^T g from c2w_window_score_backward (src/thor/score.py:28-35,
                            48-60 with grad enabled); NULL = closed-form guidance (exact_grad=False)        */
  float* cot_out;        /* mode 2 output, [frames_local, H, W, C]                                         */
  void* halo;            /* c2w_halo* or NULL.  mode 0, time-sharded: the halo PUSH is fused into this kernel — the
                            updated pixels of the first / last k owned frames are also stored into the neighbours'
                            mailboxes over NVLink and the last CTA publishes the step; complete with c2w_halo_pull  */
  int32_t halo_k;        /* Markov order k (frames per side)                                                       */
  int32_t channels;      /* C, variables per frame, 1..8 (0 = 4, the shipped configs); every count runs the same
                            kernels, instantiated per C; the fused halo push needs C = 4                           */
} c2w_guide;

/* ---- lifecycle ------------------------------------------------------------------------------------------ */
int c2w_create(const c2w_config* cfg, c2w_handle** out);
void c2w_destroy(c2w_handle* h);
const char* c2w_last_error(void);
int c2w_abi_version(void);
/* sizeof() of the structs of this header as the library was compiled, for bindings to check their own layout against:
 * which = 0 c2w_config, 1 c2w_guide, 2 c2w_adamw, 3 c2w_conv_desc, 4 c2w_point_obs; -1 for an unknown index */
int c2w_struct_size(int which);

/* ---- weights: reference state_dict entries by name (SURVEY.md §8(b)), fp32 host memory -------------------- */
int c2w_load_weight(c2w_handle* h, const char* name, const float* host_data, int64_t numel);
int c2w_finalize_weights(c2w_handle* h); /* packs to bf16 K-major [Cout, 9*Cin] and uploads; checks completeness */

/* ---- workspace ------------------------------------------------------------------------------------------- */
int64_t c2w_workspace_bytes(c2w_handle* h, int32_t max_windows);
int c2w_bind_workspace(c2w_handle* h, int32_t max_windows, void* dev_ptr, int64_t bytes);

/* Workspace variants (flags of the _ex calls; the plain calls use 0, the _vjp calls C2W_WS_VJP). */
#define C2W_WS_VJP 1          /* forward calls stash what the input-gradient pass needs                          */
#define C2W_WS_PER_SAMPLE_T 2 /* one diffusion time per sample (c2w_unet_forward_t): per-sample modulation       */
#define C2W_WS_TRAIN 4        /* training step: both of the above plus the parameter-gradient scratch             */
int64_t c2w_workspace_bytes_ex(c2w_handle* h, int32_t max_windows, int32_t flags);
int c2w_bind_workspace_ex(c2w_handle* h, int32_t max_windows, void* dev_ptr, int64_t bytes, int32_t flags);

/* VJP workspaces additionally hold the per-block stashes (LayerNorm outputs, SiLU pre-activations, qkv) and the
 * gradient buffers (about 4.5x the forward-only workspace); forward calls on them stash as they go. */
int64_t c2w_workspace_bytes_vjp(c2w_handle* h, int32_t max_windows);
int c2w_bind_workspace_vjp(c2w_handle* h, int32_t max_windows, void* dev_ptr, int64_t bytes);

/* ---- ScoreUNet.forward (model/score.py:59-70 -> model/nn.py:220-242) --------------------------------------
 * x, out: fp32 NCHW [n, C*window, H, W] on the device; scalar diffusion time t (sampling: one t per call). */
int c2w_unet_forward(c2w_handle* h, const float* x_nchw, int32_t n, float t, float* out_nchw, void* stream);
/* One diffusion time per sample, t_dev: DEVICE array of n floats (the DSM objective draws t ~ U[0,1) per sample,
 * src/thor/pipelines.py:27-35; model/score.py:61 reshapes t to [B]).  Needs a C2W_WS_PER_SAMPLE_T workspace. */
int c2w_unet_forward_t(c2w_handle* h, const float* x_nchw, int32_t n, const float* t_dev, float* out_nchw, void* stream);

/* Forcing vectors of the NEXT per-sample forward / training calls (model/score.py:63-66: emb += map_forcing(forcing)):
 * DEVICE fp32 [n, forcing_dim], one row per sample; NULL clears it.  Needs forcing_dim > 0 and a per-sample workspace
 * (C2W_WS_PER_SAMPLE_T or C2W_WS_TRAIN); the training backward also delivers map_forcing's gradients. */
int c2w_set_forcing(c2w_handle* h, const float* forcing_dev);

/* Vector-Jacobian product of ScoreUNet.forward w.r.t. x (what torch.func.jacrev / autograd computes through the UNet
 * when condition_on(exact_grad=True), src/thor/score.py:28-33,51-52): gin = (d out / d x)^T gout.  n <= max_windows
 * of a VJP workspace; out_nchw (the forward result) may be NULL. */
int c2w_unet_vjp(c2w_handle* h, const float* x_nchw, int32_t n, float t, const float* gout_nchw, float* out_nchw,
                 float* gin_nchw, void* stream);

/* ---- DefaultScoreFunction/BatchedScoreFunction.score_fn (src/thor/score.py:68-93, :111-185) ---------------
 * unfold -> UNet -> centre-pick/edge-fill compose, without materialising the unfold in fp32 or the unused
 * 12/13 of the UNet output.  traj/eps: [n_frames_local, H, W, C].  Computes windows
 * [win_first, win_first + n_win) (global indices; window j covers global frames j .. j+2k) of a trajectory with
 * n_win_global windows; local frame 0 is global frame frame_global0. */
int c2w_window_score(c2w_handle* h, const float* traj, int32_t n_frames_local, int32_t frame_global0,
                     int32_t win_first, int32_t n_win, int32_t n_win_global, float t, float* eps, void* stream);

/* Adjoint of c2w_window_score for the windows whose forward has JUST run on a VJP workspace (one chunk): compose
 * adjoint -> UNet input-gradient pass -> unfold adjoint.  cot: cotangent w.r.t. the composed score; vjp is accumulated. */
int c2w_window_score_backward(c2w_handle* h, const float* cot, int32_t n_frames_local, int32_t frame_global0,
                              int32_t win_first, int32_t n_win, int32_t n_win_global, float* vjp, void* stream);

/* The same for a SELECTION of windows (global indices, device array).  The cotangent of the composed score under the
 * coarse-graining likelihood is non-zero on the observed frames only (every t_step-th frame, exp/downscaling.py:129-132),
 * so the vector-Jacobian product of src/thor/score.py:28-33 needs the backward of ~1/t_step of the windows only.
 * c2w_window_score_sel is the forward of a selection: on a VJP workspace it stashes (n_sel <= max_windows) and is
 * followed by c2w_window_score_backward_sel; on a plain workspace it chunks like c2w_window_score.  With eps != NULL the
 * selection's part of the composed score is written into eps (same fold, by list), so the observed selection on the VJP
 * workspace and the rest on the plain one fill eps together and no window runs twice; eps == NULL stashes only.
 * pos_dev[j] = position of global window j in win_list_dev, or -1. */
int c2w_window_score_sel(c2w_handle* h, const float* traj, int32_t n_frames_local, int32_t frame_global0,
                         const int32_t* win_list_dev, int32_t n_sel, int32_t n_win_global, float t, float* eps,
                         void* stream);
int c2w_window_score_backward_sel(c2w_handle* h, const float* cot, int32_t n_frames_local, int32_t frame_global0,
                                  const int32_t* win_list_dev, const int32_t* pos_dev, int32_t n_sel, int32_t n_win_global,
                                  float* vjp, void* stream);

/* ---- layout: reference NCHW fp32 [frames, C, H, W] <-> device [frames, H, W, C] --------------------------- */
int c2w_traj_pack(const float* nchw, float* fhwc, int64_t frames, int32_t C, int32_t hw, void* stream);
int c2w_traj_unpack(const float* fhwc, float* nchw, int64_t frames, int32_t C, int32_t hw, void* stream);

/* ---- N4: normalisation fused with the layout change (data/pipeline.py:183-272) -------------------------------
 * normalize_ds + ds_to_sorted_np + packing:  fhwc[f, pix, c] = (src - shift[c]) / scale[c]
 * unnormalize_ds + np_to_ds               :  dst = fhwc[f, pix, c] * scale[c] + shift[c]
 * src / dst: fp32 per-variable arrays [C][frames][hw] (clhw != 0) or sorted-numpy order [frames][C][hw] (clhw == 0);
 * shift / scale: device fp32 [C], or per-grid-point fields [C][hw] (field != 0).  Which quantiles they are is the
 * normalisation mode (minmax / robust / robust95 / quant95 / quant99), resolved by the host. */
int c2w_normalize_pack(const float* src, float* fhwc, int64_t frames, int32_t C, int32_t hw, int32_t clhw,
                       const float* shift, const float* scale, int32_t field, void* stream);
int c2w_unpack_unnormalize(const float* fhwc, float* dst, int64_t frames, int32_t C, int32_t hw, int32_t clhw,
                           const float* shift, const float* scale, int32_t field, void* stream);

/* ---- N2 (optimiser half): torch.optim.AdamW.step() + StandardEMA.update() in one pass --------------------------
 * training_loop.py:381-390 (optimizer.step(); ema.update()), src/thor/ema.py:24-27.  All buffers: device fp32 [n]
 * (the flat parameter buffer, its gradient, the two moments, the EMA copy), 16-byte aligned; ema may be NULL.
 *   g' = g * grad_scale;  p *= 1 - lr * weight_decay;  m += (1 - beta1)(g' - m);  v = beta2 v + (1 - beta2) g'^2
 *   p -= lr / (1 - beta1^step) * m / (sqrt(v) / sqrt(1 - beta2^step) + eps);  ema = ema * ema_rate + p * (1 - ema_rate) */
typedef struct c2w_adamw {
  float lr, beta1, beta2, eps, weight_decay;
  float ema_rate;    /* StandardEMA rate (0.9999); ignored when ema == NULL */
  float grad_scale;  /* 1 / loss_scaling */
  int32_t step;      /* 1-based optimiser step count (bias correction) */
} c2w_adamw;
int c2w_adamw_ema_step(float* p, const float* g, float* m, float* v, float* ema, int64_t n, const c2w_adamw* hp,
                       void* stream);

/* ---- guided predictor / corrector (see c2w_guide) --------------------------------------------------------- */
int c2w_guided_step(const c2w_guide* g, void* stream);

/* Point observations (PointObservation in climate2weather_b200/score.py): variables observed at single grid points of
 * chosen frames, A(x)[m, c, p] = mask[m, c, p] * x[frames[m], c, rows[p], cols[p]].  The host merges the observations
 * of each (frame, pixel) into one entry, ysum = sum(mask * y) and wsum = sum(mask) per variable, so the likelihood
 * cotangent at that pixel is (ysum - wsum * x0) / var and zero elsewhere.  Entries are grouped by observed frame (slot)
 * and by strip of strip_rows full pixel rows (strip_rows * W <= C2W_POINT_STRIP_PIX), sorted by pixel within a strip. */
#define C2W_POINT_STRIP_PIX 2048
typedef struct c2w_point_obs {
  const int32_t* frame_slot; /* [own_n] observed slot of the updated frame own_lo + i, or -1                      */
  const int32_t* strip_off;  /* [n_slots * ceil(H / strip_rows) + 1] CSR offsets into the entries                */
  const int32_t* pix;        /* [n_entries] pixel index within the frame (h * W + w), unique per (slot, strip);
                              * c2w_guided_step_obs_std: runs of one pixel allowed, see there                   */
  const float* ysum;         /* [n_entries, C] sum of mask * y                                                    */
  const float* wsum;         /* [n_entries, C] number of unmasked observations                                    */
  int32_t n_slots, strip_rows;
} c2w_point_obs;
/* c2w_guided_step with the point operator: y, t_step and s_step of g are ignored, every other field keeps its meaning
 * (modes 0/1/2, vjp, cot_out, nan_flag, halo for C = 4, channels).  Mode 1 writes own_n * ceil(H / strip_rows)
 * partials. */
int c2w_guided_step_points(const c2w_guide* g, const c2w_point_obs* obs, void* stream);
/* A coarse field and point observations in one likelihood (CombinedObservation in climate2weather_b200/score.py):
 * g carries the coarse term (y, t_step, s_step, std2: c2w_guided_step), obs the point term, point_std2 (HOST, channels
 * floats) the point term's std^2 per variable; gamma is shared.  The cotangent is the sum of the two terms'.  obs is
 * built with strip_rows a multiple of s_step and strip_rows * W <= C2W_COMBINED_STRIP_PIX (the host library picks
 * s * max(1, min(H / s, floor(C2W_POINT_STRIP_PIX / (s * W))))).  Mode 1 writes own_n * ceil(H / strip_rows) partials. */
#define C2W_COMBINED_STRIP_PIX 16384
int c2w_guided_step_combined(const c2w_guide* g, const c2w_point_obs* obs, const float* point_std2, void* stream);
/* A std per observation: the guidance step of the three entry points above with each observation's own std^2.
 * g->std2 is ignored; gamma comes from g.  Coarse term: g->y and coarse_std2 (device, y's layout), both or neither.
 * Point term: obs and entry_std2 (device, [n_entries, C]), both or neither; an obs here may hold runs of entries
 * with the same pixel (consecutive, within one strip).  At least one term.  Launches K6, K6p or K6c accordingly,
 * with the argument checks of c2w_guided_step, c2w_guided_step_points or c2w_guided_step_combined. */
int c2w_guided_step_obs_std(const c2w_guide* g, const c2w_point_obs* obs, const float* coarse_std2,
                            const float* entry_std2, void* stream);
int c2w_reduce_partials(const float* partials, int32_t n, double* sumsq, void* stream);
/* x <- x - (delta eps + sqrt(2 delta) z) sigma_next, delta = tau / (sumsq / count)  (src/thor/pipelines.py:84-87).
 * z == NULL: on-chip Philox4x32-10 keyed by (seed, step_id, global pixel index). */
int c2w_corrector_update(float* x, const float* eps, const float* z, const double* sumsq, double count, float tau,
                         float sigma_next, int64_t pix0_global, int64_t npix, uint64_t seed, uint32_t step_id,
                         int32_t* nan_flag, void* stream);
/* the same for `channels` variables per pixel (1..8; 4 = the call above) */
int c2w_corrector_update_c(float* x, const float* eps, const float* z, const double* sumsq, double count, float tau,
                           float sigma_next, int64_t pix0_global, int64_t npix, int32_t channels, uint64_t seed,
                           uint32_t step_id, int32_t* nan_flag, void* stream);

/* ---- op-level hooks (parity tests of single kernels; same kernels the calls above launch) ----------------- */
/* One launch of K1 (Conv2d 3x3 pad 1, stride 1 or 2 — model/nn.py:155,157,169,185,193,194 — or a plain GEMM for the
 * 1x1 Conv1d of model/nn.py:45,47) with every epilogue option the engine uses. */
typedef struct c2w_conv_desc {
  const void* x;        /* bf16 NHWC [n_img, H, W, cin] (conv3x3) or [n_img*H*W, cin] row-major (GEMM)            */
  int32_t n_img, H, W;  /* INPUT image size                                                                       */
  int32_t cin;          /* multiple of 64                                                                         */
  int32_t stride;       /* 1 or 2 (conv3x3 only); output is [n_img, H/stride, W/stride, cout_pad]                 */
  int32_t conv3x3;      /* 0: GEMM                                                                                */
  const void* w_packed; /* bf16 [cout_pad, taps*cin], k = (r*3+s)*cin + c                                         */
  int32_t cout_pad;     /* multiple of 64                                                                         */
  const float* bias;    /* fp32 [cout_pad]                                                                        */
  int32_t mode;         /* 0 bias, 1 bias+SiLU, 2 bias+residual, 4 fp32 output                                    */
  const void* res;      /* bf16 [M, cout_pad] (mode 2; may alias out)                                             */
  void* out;            /* bf16 [M, cout_pad]                                                                     */
  float* out_f32;       /* mode 4                                                                                 */
  int32_t bn;           /* N tile (0 = pick)                                                                      */
  int32_t variant;      /* -1 pick; else bit 0: CTA pair (cta_group::2)                                            */
  int32_t max_ctas;     /* 0 = one per SM                                                                         */
  int32_t skip_loads;   /* diagnostics: stop issuing TMA loads once the ring is primed (results are garbage)      */
  void* ln_out;         /* non-NULL: fused channel LayerNorm of (bf16(out) + ln_mod) -> bf16 (bn == cout_pad)     */
  const float* ln_mod;  /* fp32 [cout_pad] or NULL                                                                */
  int32_t ln_upsample;  /* write each normalised pixel to its 2x2 block of [n_img, 2Ho, 2Wo, cout_pad]            */
  int64_t* stats;       /* diagnostics: per-CTA cycle counters [grid][12] (producer total/wait-empty, MMA total/
                           wait-full/wait-tmem, epilogue total/wait-accumulator); NULL = off                      */
} c2w_conv_desc;
int c2w_op_conv_ex(const c2w_conv_desc* d, void* stream);
/* Planning query (host only, no device call): the N-tile width the engine picks for one conv of `n_img` images on a
 * GPU with `num_sms` SMs — the wave-aware choice described in DESIGN.md (conv_pick_bn_tiled). */
int c2w_conv_tile_width(int cout_pad, int conv3x3, int n_img, int H, int W, int stride, int num_sms);
int c2w_op_conv(const void* x, int n_img, int H, int W, int cin, const void* w_packed, int cout_pad,
                const float* bias, int mode, const void* res, void* out, float* out_f32, int conv3x3, int bn,
                int max_ctas, void* stream);
int c2w_op_layernorm(const void* x_bf16, const float* mod, void* out_bf16, int64_t npix, int C, int H, int W,
                     int upsample, void* stream);
int c2w_op_attention(const void* qkv_bf16, void* out_bf16, int n, int T, int C, void* stream);
/* backward kernels of the VJP path: LayerNorm forward with its 1/std stash, LayerNorm backward (down: the forward
 * output was 2x nearest-upsampled, gy is [n, 2H, 2W, C]), attention-core backward (scratch: 2*n*T*T floats) */
int c2w_op_layernorm_inv(const void* x_bf16, const float* mod, void* out_bf16, float* inv, int64_t npix, int C,
                         void* stream);
int c2w_op_layernorm_bwd(const void* gy_bf16, const void* y_bf16, const float* inv, const void* gres_bf16,
                         void* out_bf16, int64_t npix, int C, int H, int W, int down, void* stream);
int c2w_op_attention_bwd(const void* qkv_bf16, const void* go_bf16, void* gqkv_bf16, float* scratch_2nTT, int n, int T,
                         int C, void* stream);
int c2w_op_gather_windows(const float* traj, void* out_bf16, int n, int hw, int C, int window, int cin_pad,
                          int frame0, void* stream);
int c2w_op_modulation(c2w_handle* h, float t, float* emb_out, float* mods_out, void* stream);
int c2w_total_mod_channels(c2w_handle* h);

/* ---- weight-gradient kernels (op level; the training step below launches the same kernels) ---------------------
 * c2w_op_wgrad: dW of one Conv2d 3x3 pad 1 (stride 1 or 2) or one 1x1 GEMM, the wgrad half of `fabric.backward(loss)`
 * (training_loop.py:378) — a split-K tcgen05 GEMM with K = pixels over the NHWC tensors as they are (MN-major
 * operands, no transposes), partial sums in `scratch`, deterministic reduction into
 *   dw fp32 [cout][cin][taps] (= torch's OIHW / OI1 layout, REAL channel counts), overwritten or accumulated.
 *   x  bf16 NHWC [n_img, H, W, cin_pad]  (GEMM: H = 1, W = rows per image; rows in total a multiple of 64)
 *   dy bf16 NHWC [n_img, H/stride, W/stride, cout_pad]
 *   db (may be NULL) fp32 [cout]: the conv's bias gradient, the column sums of dy, collected by the same GEMM from the
 *      dy tiles in shared memory (no second pass over dy)
 * c2w_op_colsum: out[group][c] += scale * sum over the group's rows of x[row][c] (bias gradients: one group; the
 * per-sample modulation gradients: one group per image), atomically accumulated — zero `out` first. */
int c2w_op_wgrad(const void* x, const void* dy, int32_t n_img, int32_t H, int32_t W, int32_t cin_pad, int32_t cout_pad,
                 int32_t stride, int32_t conv3x3, float* scratch, int64_t scratch_floats, float* dw, float* db,
                 int32_t cin, int32_t cout, int32_t accumulate, void* stream);
int c2w_op_colsum(const void* x_bf16, float* out, int64_t rows, int32_t C, int64_t rows_per_group, int32_t out_stride,
                  float scale, void* stream);

/* ---- training step (SURVEY.md §8(f) N2; training_loop.py:372-391, src/thor/pipelines.py:27-35) ----------------------
 * Parameter gradients of the ScoreUNet for the denoising-score-matching objective, on a C2W_WS_TRAIN workspace of
 * max_windows >= batch samples.  The flat fp32 gradient buffer holds every parameter in the order the weights were
 * loaded (the reference state_dict order), each start aligned to 4 floats: c2w_param_total floats in all,
 * c2w_param_layout(name) -> offset / numel, tensors in torch's own layouts (conv weights OIHW) — the buffer
 * climate2weather_b200.optim.AdamW steps on (c2w_adamw_ema_step) without a copy.
 *   c2w_train_forward : net(xt, t) with one diffusion time per sample (device array), stashing for the backward
 *   c2w_train_backward: gout = d loss / d prediction (fp32 NCHW) -> all parameter gradients (input-gradient convs K1,
 *                       weight-gradient GEMMs K10, bias / modulation / time-MLP sums); gin_nchw (may be NULL) receives
 *                       the gradient w.r.t. xt
 *   c2w_dsm_loss_grad : sum((out - eps)^2) and gout = 2 loss_scale (out - eps) / numel in one pass
 *   c2w_train_step    : the three calls above for one batch (loss value: *loss_sum_dev / numel * loss_scale)        */
int64_t c2w_param_total(c2w_handle* h);
/* After an optimiser step: re-pack every weight from a DEVICE copy of the parameters in the flat layout (no host round
 * trip, no re-allocation; `optimizer.step()` -> next forward, training_loop.py:384 -> :377). */
int c2w_refresh_weights(c2w_handle* h, const float* flat_params_dev, void* stream);
int c2w_param_layout(c2w_handle* h, const char* name, int64_t* offset, int64_t* numel);
int c2w_train_forward(c2w_handle* h, const float* x_nchw, int32_t n, const float* t_dev, float* out_nchw, void* stream);
int c2w_train_backward(c2w_handle* h, const float* gout_nchw, int32_t n, float* gin_nchw, float* grad_flat,
                       int32_t accumulate, void* stream);
int c2w_dsm_loss_grad(const float* out, const float* eps, float* gout, int64_t numel, float loss_scale, float* partials4096,
                      double* loss_sum_dev, void* stream);
int c2w_train_step(c2w_handle* h, const float* xt_nchw, int32_t n, const float* t_dev, const float* eps_nchw,
                   float* out_nchw, float* gout_nchw, float loss_scale, float* grad_flat, int32_t accumulate,
                   double* loss_sum_dev, void* stream);

/* ---- time-axis halo exchange over NVLink peer memory (SURVEY.md §8(e); replaces nothing in the reference, which
 * never shards a trajectory: frame i's score needs frames i-k .. i+k, src/thor/score.py:68-93) -----------------------
 * One handle per process / GPU.  c2w_halo_create allocates this rank's mailbox ([2 parities][2 sides][k frames] + step
 * counters); c2w_halo_handle exports it as a 64-byte CUDA IPC handle, which the HOST passes to the two neighbours by any
 * means (torch.distributed in the Python mirror; MPI / files for another host); c2w_halo_connect maps the neighbours'
 * mailboxes (NULL = no neighbour on that side).  c2w_halo_exchange(x_local) then refreshes the k halo frames on each
 * side of x_local [n_local_frames][frame_floats] from the neighbours' boundary frames with two small kernels on the
 * caller's stream: peer stores through NVLink + a system-scope step counter, no NCCL launch, no host synchronisation.
 * Every rank must call it the same number of times. */
typedef struct c2w_halo c2w_halo;
int c2w_halo_create(int64_t halo_bytes, c2w_halo** out);
void c2w_halo_destroy(c2w_halo* h);
int c2w_halo_handle(c2w_halo* h, void* out64);
int c2w_halo_connect(c2w_halo* h, const void* left_handle64, const void* right_handle64);
int c2w_halo_exchange(c2w_halo* h, float* x_local, int64_t n_local_frames, int64_t frame_floats, int32_t k, void* stream);
/* Fused form: c2w_guided_step(mode 0) with g->halo set does the push inside the predictor kernel; c2w_halo_pull is the
 * second half (wait for the neighbours' counters, copy the mailbox into the halo frames, advance the step).
 * c2w_halo_push_targets exposes the current slots / counters for a caller fusing the push into a kernel of its own. */
int c2w_halo_pull(c2w_halo* h, float* x_local, int64_t n_local_frames, int64_t frame_floats, int32_t k, void* stream);
int c2w_halo_push_targets(c2w_halo* h, void** slot_left, void** slot_right, void** flag_left, void** flag_right, void** done,
                          uint32_t* publish);

/* ---- measurement hooks (bench.py): kernel launches issued by this library so far; optional CUDA-event timing of
 * every forward-pass launch on its own stream, summed per class: [0] K1 conv/GEMM (tensor cores), [1] the rest --- */
int64_t c2w_launch_count(void);
/* Diagnostics build (-DC2W_DIAG, libc2w_b200_diag.so) only: per-launch {start, end} %globaltimer stamps of K1
 * (tools/timeline.py: time inside the kernels vs the gaps between them); an error in the shipped library. */
int c2w_set_timeline(c2w_handle* h, long long* buf_dev, int capacity);
int c2w_set_timing(c2w_handle* h, int enable);
int c2w_timing_read(c2w_handle* h, double* ms, int64_t* n);

#ifdef __cplusplus
}
#endif
#endif /* C2W_B200_H */
