/*
 * avc_b200.h -- C ABI of libavc_b200.so: the sm_100a kernels behind the AdaIN-VC hot path.
 *
 * The reference (jjery2243542/adaptive_voice_conversion) has no FFI: its hot path is the
 * Python class surface model.AE / solver.Solver / inference.Inferencer on top of stock
 * torch.nn modules.  Each entry point below therefore cites the reference lines (relative
 * to the reference repo root) whose torch ops it replaces; the Python side
 * (adaptive_voice_conversion_b200/model.py ...) re-exposes the reference's own class API
 * on top of these calls through ctypes.  See INTEGRATION.md for the binding.
 *
 * Conventions
 *  - plain pointers and sizes only; every pointer is a DEVICE pointer owned by the caller
 *    (PyTorch allocates; the library never allocates or frees device memory);
 *  - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing
 *    synchronises, so every call is CUDA-graph capturable;
 *  - every function returns AVC_OK (0) or a negative AVC_ERR_* code and never throws;
 *    avc_last_error() returns a static message for the most recent failure on the calling
 *    thread;
 *  - activations use the "A4" layout: a logical [B][C][T] fp32 tensor is stored as
 *    [B][C/4][T][4] (four channels interleaved per time step, C % 4 == 0), so one
 *    (sample, 4-channel chunk) is a contiguous run of T 16-byte vectors.  The reference's
 *    boundary tensors (x, dec, mu, log_sigma, eps) stay planar [B][C][T]; avc_pack_a4 /
 *    avc_unpack_a4 convert.  `*_bstride` is the distance in floats between samples, which
 *    lets a tensor be a channel sub-range of a wider one (the conv-bank concat).
 */
#ifndef AVC_B200_H_
#define AVC_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AVC_OK 0
#define AVC_ERR_INVALID (-1)     /* bad argument (null pointer, C % 4 != 0, ...) */
#define AVC_ERR_UNSUPPORTED (-2) /* valid request this kernel family does not cover */
#define AVC_ERR_CUDA (-3)        /* a CUDA runtime call failed; see avc_last_error() */

#define AVC_PAD_REFLECT 0
#define AVC_PAD_ZERO 1

#define AVC_RES_NONE 0
#define AVC_RES_SAME 1 /* out += res[t]                                   (model.py:249,368) */
#define AVC_RES_POOL 2 /* out += avg_pool1d(res, 2, ceil_mode=True)[t]    (model.py:248,319) */
#define AVC_RES_UP 3   /* out += nearest-upsample-x2(res)[t]              (model.py:61-63,367) */

/* avc_conv_desc.flags: the tensor core truncates fp32 operands to TF32; to stay unbiased the
 * TF32 path rounds to nearest -- once, where an activation is produced. */
#define AVC_F_ROUND_OUT 1 /* round out (conv block / norm_apply) or dc (norm_bwd) to TF32 */
#define AVC_F_IN_TF32 2   /* `in` is already TF32-exact: avc_conv_block_tc skips its rounding pass */
/* avc_conv_block_tc, plain stride-1 conv used as a data gradient: the epilogue also applies the
 * adjoint of the forward conv's reflect padding (pl = (flags>>8)&255, pr = (flags>>16)&255) and of
 * its residual branch (res / res_mode / res_T read as in avc_fold_desc): Tout = T+pl+pr columns are
 * computed, `out` receives the T folded time steps (what avc_fold_add_fwd produces in a second pass). */
#define AVC_F_FOLD 4
/* with AVC_F_FOLD on the persistent kernel: the epilogue also runs the backward of the UPSTREAM block's InstanceNorm /
 * AdaIN / ReLU on the folded gradient (what avc_norm_bwd does in a second pass).  The descriptor's norm, relu, eps, cond,
 * save_c, stats (inputs) and dc, dcond, dbias (outputs) then describe that upstream block -- same [B][Cout][T] shape as
 * this conv's folded output, no pixel shuffle, Cout <= 128 -- and `out` may be null when nobody else needs the folded
 * gradient itself.  dc is rounded to TF32 when AVC_F_ROUND_OUT is set. */
#define AVC_F_NORMBWD 8
#define AVC_FOLD_FLAGS(pl, pr) (AVC_F_FOLD | ((pl) << 8) | ((pr) << 16))

#define AVC_PACK_FWD 0   /* P[ci][j][co]  = W[co][ci][j]                                   */
#define AVC_PACK_DGRAD 1 /* P[co][j][ci]  = W[co][ci][K-1-j]  (transposed, tap-flipped)     */

/* One fused conv block: reflect-pad -> Conv1d -> [pixel shuffle] -> [InstanceNorm] ->
 * [AdaIN affine] -> [ReLU] -> [+ residual] -> [* mask].
 * Replaces pad_layer (model.py:21-32) + nn.Conv1d + pixel_shuffle_1d (:52-59) +
 * nn.InstanceNorm1d (:296,341) + append_cond (:77-83) + ReLU + the residual adds with
 * F.avg_pool1d / upsample (:248-249, :319-320, :366-369) of one ConvBlock.
 * With pad_mode = ZERO / in_ups = 2 the same kernel computes the data gradient of a conv
 * (see avc_fold_add_fwd).  The struct is also the argument of avc_norm_apply_fwd,
 * avc_norm_bwd. */
typedef struct avc_conv_desc {
  int32_t B, Cin, Cout, K, stride, pad_left, pad_mode, in_ups;
  int32_t Tin;  /* stored input length; logical length is Tin * in_ups (zero insertion) */
  int32_t Tout; /* conv output length */
  const float* in; /* A4 [B][Cin/4][Tin][4] */
  int64_t in_bstride;
  const float* w_packed; /* [Cin][K][w_ld] (avc_pack_conv_weight) */
  int32_t w_ld;
  const float* bias; /* [Cout] or null */
  float* out;        /* A4 [B][Cn/4][Tn][4]; Cn = Cout/(1+shuffle), Tn = Tout*(1+shuffle) */
  int64_t out_bstride;
  int32_t shuffle; /* 1: out[b][c][2t+s] = conv[b][2c+s][t] before the norm (model.py:52-59) */
  int32_t norm;    /* 1: InstanceNorm over Tn per (b, c), biased variance */
  float eps;
  int32_t relu;
  const float* cond; /* AdaIN rows: beta = cond[b*cond_bstride + c], gamma = cond[... + Cn + c]; or null */
  int64_t cond_bstride;
  const float* res; /* A4 [B][Cn/4][res_T][4] or null */
  int64_t res_bstride;
  int32_t res_mode, res_T;
  const float* mask; /* A4 like out; out *= (mask > 0); or null */
  int64_t mask_bstride;
  float* save_c; /* dense A4 [B][Cout/4][Tout][4] raw conv (+bias) kept for backward; or null */
  float* stats;  /* [B][Cn][2] = (mean, rstd) when norm; or null */
  /* ---- backward-only fields (avc_norm_bwd) ---- */
  const float* dy; /* A4 [B][Cn/4][Tn][4], grad w.r.t. the block output */
  int64_t dy_bstride;
  float* dc;    /* dense A4 [B][Cout/4][Tout][4], grad w.r.t. the raw conv output */
  float* dcond; /* [B][2*Cn] (dbeta | dgamma) rows, dcond_bstride apart; or null */
  int64_t dcond_bstride;
  float* dbias; /* [Cout], accumulated with atomics; or null */
  /* ---- tensor-core path (avc_conv_block_tc) ---- */
  const float* w_tc; /* weights packed by avc_pack_conv_weight_tc; or null */
  int32_t flags;     /* AVC_F_* */
  int32_t out_tstride, out_toff, out_T; /* avc_conv_block_tc: out time index = t*out_tstride + out_toff inside an out
                                          tensor of out_T time steps (0, 0, 0 = dense: index t of Tn) */
} avc_conv_desc;

/* Fused block forward.  norm=1 needs the whole Tn of a sample inside one CTA tile:
 * supported for Tout <= 256, otherwise AVC_ERR_UNSUPPORTED -- run it with norm=0, relu=0,
 * res=null, save_c=out-of-conv and follow with avc_norm_apply_fwd. */
int avc_conv_block_fwd(const avc_conv_desc* d, void* stream);
/* The same fused block on the tcgen05 tensor cores (TF32 inputs rounded to nearest, fp32
 * accumulation in TMEM).  Covers stride 1, in_ups 1, Cin % 16 == 0, Tout <= 256; otherwise
 * AVC_ERR_UNSUPPORTED (use avc_conv_block_fwd).  Reads d->w_tc instead of d->w_packed.
 * status: device int, set non-zero if an internal pipeline barrier timed out. */
int avc_conv_block_tc(const avc_conv_desc* d, int* status, void* stream);
/* nn.Conv1d weight [Cout][Cin][K] -> tcgen05 operand blocks (TF32-rounded), AVC_PACK_FWD or
 * AVC_PACK_DGRAD; avc_tc_packed_floats gives the buffer size for a conv with co_total output
 * and ci_total input channels (FWD: Cout, Cin; DGRAD: Cin, Cout). */
int avc_pack_conv_weight_tc(const float* w, float* packed, int Cout, int Cin, int K, int mode, void* stream);
int64_t avc_tc_packed_floats(int co_total, int ci_total, int K);
/* Diagnostics: device buffer of 4 int64 per CTA receiving clock64 at kernel start / main loop
 * done / epilogue done for subsequent avc_conv_block_tc launches (null disables). */
void avc_tc_set_debug(void* dev_buffer);
/* Same for the persistent kernel: 16 int64 per CTA: [0] start [1] end clock; wait / work cycle sums of the roles:
 * [2] producer wait-empty, [3] patch wait-full [4] patch work, [5] MMA wait-ready [6] wait-accumulator [7] issue,
 * [8] epilogue wait-accumulator [9] TMEM pass [10] parameters [11] c rows [13] out rows [14] end barrier, [12] tiles done. */
void avc_tc2_set_debug(void* dev_buffer);
/* Weight-gradient kernel: 8 int64 per CTA: [0] start [1] end clock, cycle sums [2] staging [3] wait for a free buffer
 * [4] MMA issue [5] wait for the last MMAs [6] epilogue, [7] tiles. */
void avc_wgrad_tc_set_debug(void* dev_buffer);
/* Store path of the persistent kernel's second pass (default from AVC_T2_VARIANT): bit 0 = `c` rows through bulk
 * (TMA) stores, bit 1 = `out` rows written back in place and bulk-stored. */
void avc_tc2_set_variant(int v);
/* Runtime options (process-wide; each also has an environment default read on first use):
 *   "tc_uniform_issue"  (AVC_TC_ISSUE=uniform|legacy)   tcgen05 issue loops on the uniform datapath
 *   "wgrad_reduce_v2"   (AVC_WGRAD_REDUCE=v2|v1)        unrolled partial-sum reduction of conv_wgrad_tc
 *   "tc_conv_v2"        (AVC_TC_CONV=v2|v1)             persistent, epilogue-overlapped conv block kernel (default on)
 *   "wgrad_split"       (AVC_WGRAD_KERNEL=split|r1)     weight gradient with a dedicated MMA warp, all taps in one MMA (default on)
 * avc_set_option returns AVC_ERR_INVALID for an unknown name; avc_get_option returns -1. */
int avc_set_option(const char* name, int value);
int avc_get_option(const char* name);
/* Every re-pack of a model in one launch: a DEVICE-resident table of items (null destinations
 * are skipped); max_elems = the largest destination element count in the table. */
typedef struct avc_pack_item {
  const float* w;     /* nn.Conv1d weight [Cout][Cin][K] */
  float* simt_fwd;    /* AVC_PACK_FWD   layout for avc_conv_block_fwd, or null */
  float* simt_dgrad;  /* AVC_PACK_DGRAD layout for avc_conv_block_fwd, or null */
  float* tc_fwd;      /* avc_pack_conv_weight_tc FWD layout, or null */
  float* tc_dgrad;    /* avc_pack_conv_weight_tc DGRAD layout, or null */
  float* tc_dgrad_even; /* DGRAD layout restricted to taps 0,2,4,.. (stride-2 transposed conv, even outputs), or null */
  float* tc_dgrad_odd;  /* ... taps 1,3,.. (odd outputs), or null */
  int32_t Cout, Cin, K, reserved;
} avc_pack_item;
int avc_pack_conv_weights_batch(const avc_pack_item* items_dev, int n_items, int64_t max_elems, void* stream);
/* Two-pass epilogue for long sequences: reads d->save_c, applies shuffle/norm/AdaIN/ReLU/
 * residual/mask, writes d->out and d->stats. */
int avc_norm_apply_fwd(const avc_conv_desc* d, void* stream);
/* Backward of the epilogue: dy, save_c, stats, cond -> dc, dcond, dbias.
 * (autograd of InstanceNorm1d + append_cond + ReLU, solver.py:90) */
int avc_norm_bwd(const avc_conv_desc* d, void* stream);

/* Weight gradient of pad_layer+Conv1d: dW[co][ci][j] += sum_{b,t} dc[b][co][t] *
 * xpad[b][ci][t*stride + j]  (canonical nn.Conv1d layout, accumulated with atomics into a
 * zeroed buffer).  x is the conv input A4, dc the dense grad of the raw conv output. */
typedef struct avc_wgrad_desc {
  int32_t B, Cin, Cout, K, stride, pad_left, Tin, Tout;
  const float* x;
  int64_t x_bstride;
  const float* dc; /* A4 [B][Cout/4][Tout][4], samples dc_bstride apart */
  int64_t dc_bstride;
  float* dw; /* [Cout][Cin][K] */
} avc_wgrad_desc;
int avc_conv_wgrad(const avc_wgrad_desc* d, void* stream);
/* The same gradient on the tcgen05 tensor cores (TF32 operands rounded to nearest, fp32
 * accumulate; deterministic two-stage reduction through `scratch`).  Supported for stride 1,
 * Tout % 8 == 0, Tout <= 128: avc_wgrad_tc_scratch_floats returns the scratch size in floats,
 * or -1 when the shape must use avc_conv_wgrad.  status as in avc_conv_block_tc. */
int64_t avc_wgrad_tc_scratch_floats(const avc_wgrad_desc* d);
int avc_conv_wgrad_tc(const avc_wgrad_desc* d, float* scratch, int* status, void* stream);
/* Accumulate-in-place variant (opt-in, non-deterministic summation order): every conv layer owns a
 * ZEROED buffer of avc_wgrad_acc_floats(Cout, Cin, K) floats; avc_conv_wgrad_tc_acc adds the
 * layer's weight gradient into it with vector atomics (no scratch round trip, no per-layer
 * reduction launch; d->dw is ignored) and avc_wgrad_acc_flush folds EVERY layer's buffer into its
 * nn.Conv1d gradient (dw += ...) and zeroes it again, in one launch over a DEVICE item table;
 * max_units = the largest avc_wgrad_acc_floats()/4 of the table. */
typedef struct avc_wgrad_acc_item {
  float* acc;
  float* dw; /* [Cout][Cin][K] accumulated (+=) */
  int32_t Cout, Cin, K, reserved;
} avc_wgrad_acc_item;
int64_t avc_wgrad_acc_floats(int Cout, int Cin, int K);
int avc_conv_wgrad_tc_acc(const avc_wgrad_desc* d, float* acc, int* status, void* stream);
int avc_wgrad_acc_flush(const avc_wgrad_acc_item* items_dev, int n_items, int64_t max_units, void* stream);

/* Adjoint of the reflect padding + residual adjoint.  dxp is the zero-padded "full"
 * transposed conv output (length Tin + pad_left + pad_right) produced by
 * avc_conv_block_fwd with the DGRAD weight pack; this folds the mirrored halo back
 * (adjoint of F.pad(mode='reflect'), model.py:28-30) and adds the gradient arriving
 * through the block's residual branch. */
typedef struct avc_fold_desc {
  int32_t B, C, Tin, pad_left, pad_right;
  const float* dxp; /* dense A4 [B][C/4][Tin+pad_left+pad_right][4] */
  const float* dres; /* A4 grad of the block output the residual fed; or null */
  int64_t dres_bstride;
  int32_t res_mode, res_T; /* adjoint of AVC_RES_*: SAME (res_T=Tin), POOL (res_T=ceil(Tin/2)), UP (res_T=2*Tin) */
  float* dx; /* A4 [B][C/4][Tin][4] */
  int64_t dx_bstride;
} avc_fold_desc;
int avc_fold_add_fwd(const avc_fold_desc* d, void* stream);

/* nn.Conv1d weight [Cout][Cin][K] -> kernel operand layout (AVC_PACK_*). */
int avc_pack_conv_weight(const float* w, float* packed, int Cout, int Cin, int K, int mode, void* stream);

/* planar [B][C][T] <-> A4.  add != 0 accumulates into dst instead of overwriting. */
int avc_pack_a4(const float* planar, float* a4, int64_t a4_bstride, int B, int C, int T, int round_tf32, void* stream);
int avc_unpack_a4(const float* a4, int64_t a4_bstride, float* planar, int B, int C, int T, void* stream);

/* sum over (b, t) of an A4 tensor -> out[C] (+=): bias gradient of a conv without epilogue. */
int avc_bias_grad(const float* dc, int64_t bstride, float* dbias, int B, int C, int T, void* stream);
/* The same for a tensor whose C channels are `C / group_c` layers side by side (the conv-bank gradient): channel c adds
 * into dbias_tab_dev[c / group_c][c % group_c]; dbias_tab_dev is a DEVICE array of C / group_c pointers.  One launch
 * instead of one per layer. */
int avc_bias_grad_groups(const float* dc, int64_t bstride, float* const* dbias_tab_dev, int group_c, int B, int C, int T, void* stream);

/* AdaptiveAvgPool1d(1) (model.py:231,273) and its adjoint. */
int avc_time_mean_fwd(const float* a4, int64_t bstride, float* out /*[B][C]*/, int B, int C, int T, void* stream);
int avc_time_mean_bwd(const float* dout /*[B][C]*/, float* da4, int64_t bstride, int B, int C, int T, void* stream);

/* nn.Linear (+ReLU, + residual): y_act = act(x W^T + b); out = y_act + res.
 * (model.py:252-263 dense blocks, :276 output layer, :342-343 AdaIN affine layers) */
typedef struct avc_linear_desc {
  int32_t B, N, K, relu;
  const float* x; /* [B][K] */
  int64_t x_bstride;
  const float* w;    /* [N][K] (nn.Linear layout) */
  const float* bias; /* [N] or null */
  const float* res;  /* [B][N] dense or null */
  float* y_act;      /* [B][N] dense: activation output kept for the ReLU mask; or null */
  float* out;        /* [B][N] rows out_bstride apart */
  int64_t out_bstride;
  /* backward */
  const float* dy; /* [B][N] rows dy_bstride apart */
  int64_t dy_bstride;
  const float* dx_add; /* [B][K] dense added to dx; or null */
  float* dx;           /* [B][K] dense or null */
  float* dw;           /* [N][K] accumulated (+=) */
  float* db;           /* [N] accumulated (+=) or null */
} avc_linear_desc;
int avc_linear_fwd(const avc_linear_desc* d, void* stream);
int avc_linear_bwd(const avc_linear_desc* d, void* stream); /* mask = (y_act > 0) when relu */

/* The SpeakerEncoder tail as one kernel per direction (model.py:252-263 dense_blocks, :273-276
 * output_layer): n_blocks x { y = relu(W1 h + b1); a = relu(W2 y + b2); h = a + h }, out = Wo h + bo.
 * Built for C = c_out = 128 (AVC_ERR_UNSUPPORTED otherwise: use avc_linear_fwd/bwd per layer).
 * params: DEVICE table of 4*n_blocks+2 pointers [W1_l, b1_l]* [W2_l, b2_l]* Wo bo (nn.Linear layouts).
 * save  : [3*n_blocks+1][B][C] planes h_0..h_n | y_0.. | a_0.. (null at inference).
 * gsave : [2*n_blocks+1][B][C] planes g1_0.. | g2_0.. | dout: the ReLU-masked upstream gradient of
 *         every linear layer = left operand of its weight gradient (avc_linear_batch_dw). */
typedef struct avc_dense_stack_desc {
  int32_t B, C, c_out, n_blocks;
  const float* const* params;
  const float* x; /* [B][C] */
  float* save;
  float* out;        /* [B][c_out] */
  const float* dout; /* [B][c_out] (backward) */
  float* gsave;
  float* dx; /* [B][C] */
} avc_dense_stack_desc;
int avc_dense_stack_fwd(const avc_dense_stack_desc* d, void* stream);
int avc_dense_stack_bwd(const avc_dense_stack_desc* d, void* stream);

/* L same-shape nn.Linear layers per launch (the 12 AdaIN affine layers model.py:342-343; the weight
 * gradients of the dense stack).  Layer l reads x + x_off[l] ([B][K], rows x_bstride apart) and
 * reads/writes the [B][N] tensor at y_off[l] (rows y_bstride apart): `out` in _fwd, the upstream
 * gradient `y` in _dx/_dw.  params / grads: DEVICE tables [W_l, b_l]* / [dW_l, db_l]* (accumulated).
 * _dx: dx[B][K] = sum_l y_l W_l (+ dx_add) through the scratch part[L][B][K]. */
#define AVC_LINEAR_BATCH_MAX 16
typedef struct avc_linear_batch_desc {
  int32_t L, B, N, K;
  const float* const* params;
  float* const* grads;
  const float* x;
  int64_t x_off[AVC_LINEAR_BATCH_MAX];
  int64_t x_bstride;
  const float* y;
  float* out;
  int64_t y_off[AVC_LINEAR_BATCH_MAX];
  int64_t y_bstride;
  float* part;
  const float* dx_add;
  float* dx;
} avc_linear_batch_desc;
int avc_linear_batch_fwd(const avc_linear_batch_desc* d, void* stream);
int avc_linear_batch_dx(const avc_linear_batch_desc* d, void* stream);
int avc_linear_batch_dw(const avc_linear_batch_desc* d, void* stream);

/* VAE reparameterisation (model.py:383-384) fused with the A4->planar conversion of the
 * two heads: z = mu + exp(log_sigma/2)*eps (eps null: z = mu, the inference path :389-390). */
int avc_reparam_fwd(const float* mu4, const float* ls4, const float* eps /*planar or null*/,
                    float* mu /*planar or null*/, float* ls /*planar or null*/, float* z4,
                    int B, int C, int T, void* stream);
/* dmu4 = dz4 + dmu_ext ; dls4 = dz4 * eps * 0.5*exp(ls/2) + dls_ext  (ext planar or null) */
int avc_reparam_bwd(const float* dz4, const float* ls4, const float* eps, const float* dmu_ext,
                    const float* dls_ext, float* dmu4, float* dls4, int B, int C, int T, void* stream);

/* Losses of Solver.ae_step (solver.py:84-88) with their gradients in one pass.
 * hp (device): [0]=lambda_rec [1]=lambda_kl.  sums (device, zeroed by the call):
 * [0]=sum|dec-x| [1]=sum(exp(ls)+mu^2-1-ls).  d* receive d(lambda_rec*L1 + lambda_kl*KL). */
int avc_vae_loss(const float* dec, const float* x, int64_t n_rec, const float* mu, const float* ls,
                 int64_t n_lat, const float* hp, float* sums, float* ddec, float* dmu, float* dls,
                 void* stream);

/* clip_grad_norm_ + Adam(amsgrad, L2 weight decay) over flat fp32 buffers
 * (solver.py:91-93, :75-77).  avc_sqnorm writes sum(g^2) to out[0] (deterministic
 * two-stage reduction; scratch >= 1024 floats).
 * hp (device): [2]=grad_scale (1/world for DP) [3]=lr [4]=beta1 [5]=beta2 [6]=eps
 * [7]=weight_decay [8]=max_norm [9]=amsgrad(0/1).  step (device, float) is incremented by
 * the kernel.  The clip coefficient is min(1, max_norm / (grad_scale*sqrt(sqnorm) + 1e-6)). */
int avc_sqnorm(const float* g, int64_t n, float* scratch, float* out, void* stream);
int avc_adam_step(float* p, const float* g, float* m, float* v, float* vmax, int64_t n,
                  const float* hp, const float* sqnorm, float* step, void* stream);

int avc_fill_zero(void* ptr, int64_t bytes, void* stream);

/* Spectral normalisation of the decoder layers (torch.nn.utils.spectral_norm, dim=0, one power
 * iteration, eps=1e-12; model.py:334-344 with sn: True).  One item per layer, Wm = w_orig viewed as
 * [rows][cols] (rows = Cout, cols = Cin*K or in_features).  Both calls take a DEVICE-resident item
 * table and run one CTA per item; every reduction has a fixed order (no atomics), so u, v, sigma and
 * the outputs are bit-identical run to run.
 * avc_spectral_norm_fwd, update != 0 (module.training): v = normalize(Wm^T u), u = normalize(Wm v)
 *   (normalize(x) = x / max(|x|, 1e-12)), written back to u / v; then sigma = u . (Wm v) and
 *   w_sn = w_orig / sigma.  update == 0: sigma from the stored u, v; u and v are not written.  grad is
 *   not read.
 * avc_spectral_norm_bwd: grad holds dL/dw_sn on entry and dL/dw_orig on return (u, v constants):
 *   grad = (grad - <grad, w_sn> u v^T) / sigma, with the sigma / w_sn of the last forward. */
typedef struct avc_sn_item {
  const float* w_orig; /* [rows][cols] */
  float* w_sn;         /* [rows][cols] w_orig / sigma */
  float* u;            /* [rows] */
  float* v;            /* [cols] */
  float* sigma;        /* [1] */
  float* grad;         /* [rows][cols], backward only (may be null for the forward) */
  int32_t rows, cols;
} avc_sn_item;
int avc_spectral_norm_fwd(const avc_sn_item* items_dev, int n_items, int update, void* stream);
int avc_spectral_norm_bwd(const avc_sn_item* items_dev, int n_items, void* stream);

/* tcgen05 self-test (one CTA): D[128][N] = sum_k A_k * B_k^T over nk K=8 tf32 steps, the
 * operands given as raw shared-memory images; strides[10] = {a_lbo, a_sbo, b_lbo, b_sbo,
 * a_kstep, b_kstep, a_off, b_off (bytes), a_layout, b_layout (UMMA swizzle code, 0 = none)}; a_mn/b_mn = 1 for MN-major operands; the nk steps
 * are issued `reps` times (accumulating) for timing.  status (device int[2]): [0] non-zero if
 * the completion barrier timed out, [1] SM cycles from first MMA issue to completion.  Used by the tests to
 * pin the UMMA descriptor conventions the conv kernels rely on. */
int avc_tc_probe_gemm(const float* a_img, int a_bytes, const float* b_img, int b_bytes, const uint32_t* strides,
                      int nk, int N, int a_mn, int b_mn, int reps, float* D, int* status, void* stream);
/* Read-back variant of the self-test: the accumulator is read with 16-column tcgen05.ld's starting at
 * column `shift` + 16 j (any shift >= 0; columns below `shift` are left untouched in D). */
void avc_tc_probe_set_ld_shift(int shift);
/* Store-path probe (diagnostic): `ctas` CTAs of 256 threads each write bytes_per_cta (multiple of 4096) to their own
 * region of dst; mode 0 = STG.128, 1 = 2 KB bulk (TMA) stores from shared memory, 2 = half each; cycles[cta] = span. */
int avc_probe_store(float* dst, long long bytes_per_cta, int ctas, int mode, long long* cycles, void* stream);

const char* avc_last_error(void);
/* "sm_100a" build tag, number of kernels launched so far by this process (for bench.py's
 * gpu_launches claim). */
const char* avc_build_info(void);
int64_t avc_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* AVC_B200_H_ */
