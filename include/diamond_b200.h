/* diamond_b200 — C ABI of the B200-native DIAMOND hot path (libdiamond_b200.so).
 *
 * The reference (eloialonso/diamond @ 5bcd159) is pure Python and has no FFI of its own (SURVEY.md section 8b); the
 * seam is its Python module surface.  Every entry point below therefore names the reference call site it replaces.
 * The Python mirror in diamond_b200/ binds these with ctypes (see INTEGRATION.md for the stub a maintainer adds).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host; activations are fp32
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous on it, never synchronise the device and never
 *     allocate on the hot path (the caller owns every buffer, including the workspace)
 *   - return value 0 = ok; nonzero = error, message via dmd_last_error() (thread-local)
 *   - one host thread per GPU (the reference is one process per rank, src/main.py:26)
 */
#ifndef DIAMOND_B200_H_
#define DIAMOND_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DMD_VERSION 100

int dmd_version(void);
const char* dmd_last_error(void);
/* Number of kernels launched by this library on the calling thread since the last reset (bench.py gpu_launches). */
long long dmd_launch_count(int reset);
/* Diagnostics: in-stream kernel trace.  Between dmd_ktrace_begin(capacity) and dmd_ktrace_end every conv / prep / attention /
 * wrap launch issued by this library (also into a CUDA graph being captured) gets a slot and stores the GPU nanosecond timer
 * when its inputs are ready; dmd_ktrace_end (after a device synchronisation) copies the stamps out and returns their count,
 * dmd_ktrace_name(i) describes launch i.  Differences of consecutive stamps are the in-graph kernel durations
 * (scripts/ktrace.py).  Not thread-safe; off (null slots, one predicated test per kernel) unless begun. */
int dmd_ktrace_begin(int capacity);
int dmd_ktrace_end(long long* stamps, int capacity);
const char* dmd_ktrace_name(int i);

/* ---------------------------------------------------------------------------------------------------------------
 * Per-op entry points (NHWC fp32 activations).
 * ------------------------------------------------------------------------------------------------------------- */

/* Replaces nn.Conv2d weight use (src/models/blocks.py:18-19,96): packs a torch-layout weight [Cout][CinReal][k][k]
 * into the fp16 tensor-core operand layout [taps][Cin/8][CoutPad][8].  c0_real/c0_store describe a zero-padded first
 * source (e.g. 15 real channels stored as a 16-channel operand); for an unpadded source pass c0_real = c0_store = CinReal. */
int dmd_pack_conv_weight(const float* w, void* wpk, int Cout, int CoutPad, int CinReal, int Cin, int taps,
                         int c0_real, int c0_store, int precise, void* stream);
/* precise = 1: split-fp16 packing [W_hi | W_hi | W_lo] (3*Cin channels per tap) for dmd_conv_desc.precise convs: the
 * product is evaluated as A_hi W_hi + A_lo W_hi + A_hi W_lo on the tensor cores, i.e. to ~2^-22 instead of 2^-11.  Used
 * for the layers whose input is the raw residual stream (1x1 skip projections, conv_in) and for conv_out.
 * precise = 3: the tap-row-stacked layout [dy][Cin/8][3*CoutPad][8] of 3x3 kernels (dmd_conv_desc.wpk_layout = 1): one
 * tensor-core instruction per kernel ROW with N = 3*CoutPad, the dx shift applied on the output side (conv_tc.cuh). */

/* Activation operand ("PLC16": padded-linear, chunk-major fp16; layout in diamond_b200/csrc/conv_tc.cuh).  One pass over
 * an NHWC fp32 tensor applies what the reference runs on a conv INPUT — GroupNorm (blocks.py:28) or AdaGroupNorm
 * (blocks.py:41-45), SiLU (blocks.py:143-144), channel concat as two sources (blocks.py:174), nearest-2x upsample
 * (blocks.py:109) — and writes the operand(s) the convolution consumes. */
size_t dmd_plc16_bytes(int B, int H, int W, int C);   /* H, W: conv input size (after upsampling) */

typedef struct dmd_prep_desc {
  const float* src0;     /* NHWC [B][Hs][Ws][C0] */
  const float* src1;     /* NHWC [B][Hs][Ws][C1] or NULL */
  int C0, C1;            /* multiples of 8 */
  int B, Hs, Ws;
  int upsample;          /* 0 none ; 1 nearest-2x (blocks.py:109) ; 2 zero insertion (adjoint of the stride-2 subsample) */
  int mode;              /* 0 raw ; 1 AdaGroupNorm ; 2 affine GroupNorm */
  int silu;
  const double* stats0;  /* [B][C0/gs0][2] (sum, sumsq) */
  const double* stats1;
  int gs0, gs1;
  const float* film;     /* [B][film_stride] ; scale at film_off + c, shift at film_off + (C0+C1) + c */
  int film_stride, film_off;
  const float* gamma;    /* [C0+C1] */
  const float* beta;
  float eps;
  void* dst0;            /* operand of src0: dmd_plc16_bytes(B, H, W, C0) */
  void* dst1;
  void* dst_raw0;        /* optional: the un-normalised operand as well (1x1 skip projection, blocks.py:133,142) */
  void* dst_raw1;
  void* dst_lo0;         /* optional low parts (split-fp16): fp16(y - fp16(y)) of the transformed operand ... */
  void* dst_lo1;
  void* dst_raw_lo0;     /* ... and of the raw operand */
  void* dst_raw_lo1;
} dmd_prep_desc;

int dmd_prep_act(const dmd_prep_desc* d, void* stream);

typedef struct dmd_conv_desc {
  const void* src0;      /* PLC16 operand, C0 channels */
  const void* src1;      /* second operand (channel concat) or NULL */
  int C0, C1;            /* multiples of 16 */
  int B, H, W;           /* conv input size */
  int taps;              /* 9 = 3x3 pad 1 ; 1 = 1x1 */
  int stride;            /* 1 or 2 (blocks.py:96) */
  const void* wpk;       /* from dmd_pack_conv_weight */
  const float* bias;     /* [Cout] or NULL */
  int Cout, CoutPad;     /* CoutPad: multiple of 16, <= 128 */
  const float* residual; /* NHWC like out, or NULL (blocks.py:145) */
  float* out;            /* NHWC [B][Ho][Wo][Cout] */
  double* out_stats;     /* [B][Cout/out_gs][2], accumulated (caller zeroes) or NULL */
  int out_gs;
  int debug;             /* bring-up only; 0 */
  void* debug_buf;       /* bring-up only; NULL */
  int precise;           /* 1: split-fp16 (needs src*_lo and weights packed with precise = 1) */
  int wpk_layout;        /* 0: tap-major weights ; 1: tap-row-stacked (dmd_pack_conv_weight precise = 3; 3x3, non-split only) */
  const void* src0_lo;
  const void* src1_lo;
  /* Optional fused 1x1 projection accumulated into the same output: out += W_x . cat(x0, x1) + b_x  (the skip path
   * r = proj(x) of ResBlock.forward, blocks.py:142,145).  Operands are split-fp16 (hi + lo), weights packed with taps = 1,
   * precise = 1. */
  const void* xsrc0; const void* xsrc1; const void* xsrc0_lo; const void* xsrc1_lo;
  int xC0, xC1;
  const void* wpk_x;
  const float* bias_x;
} dmd_conv_desc;

int dmd_conv2d_fprop(const dmd_conv_desc* d, void* stream);

/* Backward-data of nn.Conv2d = dmd_conv2d_fprop on dL/dy with the weights transposed and the taps flipped: packs
 * w'[ci][co][t'] = w[co][ci_off + ci][taps-1-t'] of a torch weight [CoutF][CinTotF][k][k] for the CinK input channels starting
 * at ci_off (one call per source of a channel concat) into [taps][round16(CoutF)/8][round16(CinK)][8] fp16. */
int dmd_pack_conv_weight_dgrad(const float* w, void* wpk, int CoutF, int CinTotF, int ci_off, int CinK, int taps, void* stream);

/* Backward-filter of nn.Conv2d (torch autograd conv2d_weight; reference forward src/models/blocks.py:18-19,96,109-110) on
 * tcgen05: dW[co][ci_off+ci][t] (+)= inv_scale * sum_q GY[q][co] * X[q + o_t][ci] over the padded-linear positions of the
 * two PLC16 operands (layout and kernel: diamond_b200/csrc/wgrad_tc.cuh).  Deterministic: per-CTA partial sums are reduced in
 * a fixed order.  A stride-2 conv passes its gradient zero-inserted (dmd_prep_desc.upsample = 2) at the conv INPUT size. */
typedef struct dmd_wgrad_desc {
  const void* grad;      /* PLC16 operand of dL/dy: Cg stored channels (multiple of 8, <= 64), Cout real */
  const void* act;       /* PLC16 operand of the conv input: Ca stored channels (16 / 32 / 64), Cin real */
  int Cg, Ca;
  int B, H, W;           /* conv input size */
  int taps;              /* 9 or 1 */
  float* dW;             /* torch layout [Cout][CinTot][taps] fp32 */
  int Cout, Cin, CinTot, ci_off;
  const float* inv_scale; /* device scalar multiplied into the result, or NULL */
  int accumulate;        /* dW += instead of dW = */
  void* partial;         /* workspace of dmd_wgrad_partial_bytes() */
  size_t partial_bytes;
  int debug;             /* bring-up only; 0 */
} dmd_wgrad_desc;
size_t dmd_wgrad_partial_bytes(void);
int dmd_conv2d_wgrad(const dmd_wgrad_desc* d, void* stream);

/* Host-only twins of dmd_conv2d_fprop / dmd_prep_act: run exactly the same validation and planning, touch neither the
 * device nor the pointed-to memory (pointers are only tested for NULL), and report the launch plan.  They make the
 * shape limits and the error behaviour (return code + dmd_last_error()) testable without a GPU. */
typedef struct dmd_conv_plan_info {
  int tiles;             /* 128-row tiles (one CTA per SM walks a contiguous range of them) */
  int kslabs;            /* 16-channel K slabs per tile, fused projection included */
  int stages;            /* depth of the shared-memory slab ring */
  int tmem_cols;         /* TMEM columns per accumulator (two are allocated) */
  unsigned long long smem_bytes;    /* dynamic shared memory of the launch */
  unsigned long long weight_bytes;  /* resident packed weights */
} dmd_conv_plan_info;
int dmd_conv_plan(const dmd_conv_desc* d, dmd_conv_plan_info* out);
int dmd_prep_plan(const dmd_prep_desc* d, int* blocks, int* pos_per_block, int* sources);

/* GroupNorm partial sums of an NHWC tensor: stats[n][g] += (sum, sumsq) (blocks.py:28,43). */
int dmd_gn_stats(const float* x, double* stats, int B, int HW, int C, int gs, void* stream);

/* SelfAttention2d.forward (blocks.py:62-72), L = H*W <= 64 tokens, C <= 64, head_dim 8. */
int dmd_attn_fwd(const float* x, const double* stats_in, const float* gamma, const float* beta, const float* wqkv,
                 const float* bqkv, const float* wout, const float* bout, float* out, double* out_stats, int B, int L,
                 int C, int gs, float eps, void* stream);

int dmd_nchw_to_nhwc(const float* in, float* out, int B, int C, int CP, int HW, void* stream);
int dmd_nhwc_to_nchw(const float* in, float* out, int B, int C, int CP, int HW, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Denoiser executor: InnerModel.forward (inner_model.py:44-49) + Denoiser.denoise (denoiser.py:86-91) +
 * DiffusionSampler.sample (diffusion_sampler.py:31-58) as one plan of kernels, replayed as a CUDA graph.
 * ------------------------------------------------------------------------------------------------------------- */
#define DMD_MAX_LEVELS 8

typedef struct dmd_denoiser_config {
  int img_channels;             /* InnerModelConfig.img_channels */
  int num_steps_conditioning;   /* frame stack */
  int cond_channels;
  int num_levels;
  int depths[DMD_MAX_LEVELS];
  int channels[DMD_MAX_LEVELS];
  int attn_depths[DMD_MAX_LEVELS];
  int num_actions;
  float sigma_data;             /* DenoiserConfig */
  float sigma_offset_noise;
} dmd_denoiser_config;

typedef struct dmd_denoiser dmd_denoiser;

dmd_denoiser* dmd_denoiser_create(const dmd_denoiser_config* cfg);
void dmd_denoiser_destroy(dmd_denoiser* h);

/* Number of parameter/buffer tensors expected by dmd_denoiser_set_weights == len(InnerModel.state_dict()). */
int dmd_denoiser_num_tensors(const dmd_denoiser* h);
/* Bytes of device memory needed for packed weights (caller allocates, passes to set_weights). */
size_t dmd_denoiser_packed_bytes(const dmd_denoiser* h);
/* ptrs_host: host array of device pointers, in InnerModel.state_dict() order (fp32, torch layouts).
 * Re-packs the tensor-core copies; call again after every optimizer step / load_state_dict. */
int dmd_denoiser_set_weights(dmd_denoiser* h, const float* const* ptrs_host, int n_ptrs, void* packed, void* stream);

/* H, W need not be multiples of 2^(levels-1): like UNet.forward (blocks.py:225-229,245) the executor zero-pads the conv_in
 * output at the bottom / right, runs the U-Net on the padded size and crops before norm_out / conv_out (inference entry
 * points; the training entry points reject such sizes).  The deepest level must hold 64 positions when it has attention. */
size_t dmd_denoiser_workspace_bytes(const dmd_denoiser* h, int B, int H, int W);

/* One Denoiser.denoise / compute_model_output call.  noisy (B,C,H,W), sigma (B) or (1), obs (B,T*C,H,W),
 * act (B,T) int64.  out_model / out_denoised are NCHW (B,C,H,W); either may be NULL. */
int dmd_denoiser_forward(dmd_denoiser* h, int B, int H, int W, const float* noisy, const float* sigma,
                         int sigma_is_scalar, const float* obs, const int64_t* act, float* out_model,
                         float* out_denoised, void* workspace, size_t workspace_bytes, void* stream);

/* InnerModel.forward (inner_model.py:44-49): inputs already rescaled by the caller (denoiser.py:75-76), c_noise (B) or
 * (1).  out: (B,C,H,W) NCHW model output. */
int dmd_inner_model_forward(dmd_denoiser* h, int B, int H, int W, const float* noisy_rescaled, const float* c_noise,
                            int c_noise_is_scalar, const float* obs_rescaled, const int64_t* act, float* out,
                            void* workspace, size_t workspace_bytes, void* stream);

/* ---- Training (Denoiser.forward + loss.backward(), src/models/diffusion/denoiser.py:93-122, src/trainer.py:365-366).
 * dmd_inner_model_forward_train = dmd_inner_model_forward that keeps every activation (and the GroupNorm statistics) in the
 * training workspace; dmd_denoiser_backward consumes them: given dL/d(model output) (B,C,H,W) it writes the gradient of
 * EVERY parameter into one flat fp32 buffer (16-byte aligned slices, layout from dmd_denoiser_grad_layout, state_dict
 * order; buffers such as noise_emb.weight get zeros).  Convolutions run on tcgen05 (dgrad = fprop with transposed weights,
 * wgrad = dmd_conv2d_wgrad), gradients carry a power-of-two loss scale chosen from max|grad_out| on the device.  The flat
 * buffer is what a data-parallel step all-reduces in ONE collective (utils.py:105-106 wraps each model in DDP instead). */
size_t dmd_denoiser_train_workspace_bytes(const dmd_denoiser* h, int B, int H, int W);
/* offsets / numels: n = dmd_denoiser_num_tensors entries (floats); returns the total length of the flat buffer. */
long long dmd_denoiser_grad_layout(const dmd_denoiser* h, long long* offsets, long long* numels, int n);
int dmd_inner_model_forward_train(dmd_denoiser* h, int B, int H, int W, const float* noisy_rescaled, const float* c_noise,
                                  int c_noise_is_scalar, const float* obs_rescaled, const int64_t* act, float* out,
                                  void* workspace, size_t workspace_bytes, void* stream);
int dmd_denoiser_backward(dmd_denoiser* h, int B, int H, int W, const float* grad_out, float* grads, long long grads_numel,
                          void* workspace, void* stream);

typedef struct dmd_sampler_config {
  int num_sigmas;               /* len(self.sigmas) = num_steps_denoising + 1, last one 0 */
  const float* sigmas_host;     /* host array, fp32 values of DiffusionSampler.sigmas */
  int order;                    /* 1 Euler, 2 Heun */
  float s_churn, s_tmin, s_tmax, s_noise;
} dmd_sampler_config;

/* DiffusionSampler.sample (src/models/diffusion/diffusion_sampler.py:31-58), whole loop in one call, replayed as a CUDA graph.
 * Every buffer is used IN PLACE (no staging copies; a graph is cached per distinct set of addresses):
 *   traj  (num_sigmas, B, C, H, W): slot 0 holds the initial x ~ N(0,1) on entry (drawn by the CALLER with torch so that RNG
 *         streams match the reference, :36); slot i+1 receives the iterate after step i (the reference's `trajectory`).
 *   eps   (num_steps, B, C, H, W) churn noise (:42) or NULL.
 *   out_x (B, C, H, W) or NULL: additionally receives the final iterate (e.g. a slot of the caller's frame ring).
 *   ring_head = -1: prev_obs (B, T*C, H, W), prev_act (B, T) as the reference passes them.
 *   ring_head >= 0: the WorldModelEnv's resident buffers -- prev_obs = frames (T, B, C, H, W), prev_act = actions (T, B), where
 *         LOGICAL slot k (0 = oldest) is physical slot (ring_head + k) % T: the per-step `roll` of both buffers
 *         (src/envs/world_model_env.py:74-75) becomes an index increment.
 * The conditioning path (Fourier + action embedding -> MLP -> all FiLM linears) of all denoising steps is evaluated once, up
 * front: the sigma schedule is host-known (:27) and the actions are fixed during a call. */
int dmd_sampler_sample(dmd_denoiser* h, const dmd_sampler_config* sc, int B, int H, int W, const float* prev_obs,
                       const int64_t* prev_act, int ring_head, float* traj, const float* eps, float* out_x, void* workspace,
                       size_t workspace_bytes, int use_graph, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Actor-critic executor: ActorCritic.predict_act_value (src/models/actor_critic.py:68-73) = ActorCriticEncoder
 * (:101-113: Conv3x3 + [SmallResBlock (blocks.py:116-123), MaxPool2d]*) -> flatten -> LSTMCell -> actor / critic heads.
 * ------------------------------------------------------------------------------------------------------------- */
typedef struct dmd_actor_critic_config {
  int lstm_dim;
  int img_channels;
  int img_size;
  int num_levels;
  int channels[DMD_MAX_LEVELS];
  int down[DMD_MAX_LEVELS];
  int num_actions;
} dmd_actor_critic_config;

typedef struct dmd_actor_critic dmd_actor_critic;

dmd_actor_critic* dmd_actor_critic_create(const dmd_actor_critic_config* cfg);
void dmd_actor_critic_destroy(dmd_actor_critic* h);
int dmd_actor_critic_num_tensors(const dmd_actor_critic* h);          /* == len(ActorCritic.state_dict()) */
size_t dmd_actor_critic_packed_bytes(const dmd_actor_critic* h);
int dmd_actor_critic_set_weights(dmd_actor_critic* h, const float* const* ptrs_host, int n_ptrs, void* packed, void* stream);
size_t dmd_actor_critic_workspace_bytes(const dmd_actor_critic* h, int B);
/* obs (B,C,S,S) NCHW; hx_in/cx_in (B,lstm_dim); outputs: logits (B,A), val (B), hx_out/cx_out (B,lstm_dim). */
int dmd_actor_critic_forward(dmd_actor_critic* h, int B, const float* obs, const float* hx_in, const float* cx_in,
                             float* logits, float* val, float* hx_out, float* cx_out, void* workspace,
                             size_t workspace_bytes, void* stream);

/* ---- Actor-critic training: ActorCritic.predict_act_value under autograd (src/models/actor_critic.py:68-73; the imagined
 * rollout calls it with grad, src/coroutines/env_loop.py:31,57, and src/trainer.py:366 back-propagates through time).
 * dmd_actor_critic_forward leaves every activation in its workspace; ONE dmd_actor_critic_backward call is one node of the
 * BPTT graph: given the gradients wrt (logits, val, hx_out, cx_out) (any may be NULL = zero) it writes the gradients wrt
 * (hx_in, cx_in) and the gradient of every parameter into a flat fp32 buffer (layout: dmd_actor_critic_grad_layout).
 * `workspace` is the forward's (untouched since); `scratch` is transient and may be shared by all nodes of a stream. */
size_t dmd_actor_critic_backward_scratch_bytes(const dmd_actor_critic* h, int B);
long long dmd_actor_critic_grad_layout(const dmd_actor_critic* h, long long* offsets, long long* numels, int n);
int dmd_actor_critic_backward(dmd_actor_critic* h, int B, const float* hx_in, const float* cx_in, const float* hx_out,
                              const float* g_logits, const float* g_val, const float* g_hx, const float* g_cx, float* grads,
                              long long grads_numel, float* g_hx_in, float* g_cx_in, void* workspace, void* scratch,
                              size_t scratch_bytes, void* stream);
/* Same, but ADDS the parameter gradients to what `grads` already holds: the nodes of one back-propagation-through-time pass
 * accumulate into one flat buffer (what autograd's AccumulateGrad does tensor by tensor in the reference, trainer.py:366). */
int dmd_actor_critic_backward_accumulate(dmd_actor_critic* h, int B, const float* hx_in, const float* cx_in, const float* hx_out,
                                         const float* g_logits, const float* g_val, const float* g_hx, const float* g_cx,
                                         float* grads, long long grads_numel, float* g_hx_in, float* g_cx_in, void* workspace,
                                         void* scratch, size_t scratch_bytes, void* stream);

/* compute_lambda_returns (src/models/actor_critic.py:116-143): rew / val_bootstrap fp32 [B][T], end / trunc int64 [B][T] ->
 * out fp32 [B][T]; one thread per environment walks time backwards; bit-identical to the reference's torch expression. */
int dmd_lambda_returns(const float* rew, const int64_t* end, const int64_t* trunc, const float* val_bootstrap, float* out, int B,
                       int T, double gamma, double lambda_, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Reward / termination model: RewEndModel.predict_rew_end (src/models/rew_end_model.py:42-55; SURVEY.md 8 f1), called once
 * per imagined step (src/envs/world_model_env.py:97) and over the burn-in frames of each fresh episode (:120-129).
 * ------------------------------------------------------------------------------------------------------------- */
typedef struct dmd_rew_end_config {
  int lstm_dim;
  int img_channels;
  int img_size;
  int cond_channels;
  int num_levels;
  int depths[DMD_MAX_LEVELS];
  int channels[DMD_MAX_LEVELS];
  int attn_depths[DMD_MAX_LEVELS];
  int num_actions;
} dmd_rew_end_config;
typedef struct dmd_rew_end dmd_rew_end;
dmd_rew_end* dmd_rew_end_create(const dmd_rew_end_config* cfg);
void dmd_rew_end_destroy(dmd_rew_end* h);
int dmd_rew_end_num_tensors(const dmd_rew_end* h);           /* == len(RewEndModel.state_dict()) */
size_t dmd_rew_end_packed_bytes(const dmd_rew_end* h);
int dmd_rew_end_set_weights(dmd_rew_end* h, const float* const* ptrs_host, int n_ptrs, void* packed, void* stream);
size_t dmd_rew_end_workspace_bytes(dmd_rew_end* h, int rows);  /* rows = b * t */
/* obs / next_obs (b, t, C, S, S), act (b, t) int64, hx_in / cx_in (b, lstm_dim) or NULL (zero state).
 * logits_rew (b, t, 3), logits_end (b, t, 2), hx_out / cx_out (b, lstm_dim). */
int dmd_rew_end_predict(dmd_rew_end* h, int b, int t, const float* obs, const float* next_obs, const int64_t* act,
                        const float* hx_in, const float* cx_in, float* logits_rew, float* logits_end, float* hx_out,
                        float* cx_out, void* workspace, size_t workspace_bytes, void* stream);

/* ---- Reward / termination training: RewEndModel.forward under autograd (src/models/rew_end_model.py:57-90; trained in
 * turn with the denoiser and the actor-critic, src/trainer.py:349-388).  dmd_rew_end_forward_train = predict_rew_end from a
 * zero LSTM state that keeps every activation (encoder, the gates and cell states of all t LSTM steps, head input) in the
 * training workspace, on a plan of its own: a later dmd_rew_end_predict is unaffected.  dmd_rew_end_backward consumes
 * them: given dL/dlogits it writes (assigns) the gradient of EVERY parameter into one flat fp32 buffer (16-byte aligned
 * slices in state_dict order, layout from dmd_rew_end_grad_layout).  The head and the LSTM backward run in fp32; the
 * encoder backward on tcgen05 with a power-of-two loss scale chosen on the device from max|dL/dfeatures|. */
size_t dmd_rew_end_train_workspace_bytes(dmd_rew_end* h, int b, int t);   /* 0 (dmd_last_error) when b, t are invalid */
long long dmd_rew_end_grad_layout(const dmd_rew_end* h, long long* offsets, long long* numels, int n);
/* obs / next_obs (b, t, C, S, S) fp32, act (b, t) int64 -> logits_rew (b, t, 3), logits_end (b, t, 2). */
int dmd_rew_end_forward_train(dmd_rew_end* h, int b, int t, const float* obs, const float* next_obs, const int64_t* act,
                              float* logits_rew, float* logits_end, void* workspace, size_t workspace_bytes, void* stream);
/* g_logits_rew (b, t, 3), g_logits_end (b, t, 2); `workspace` is the forward's, untouched since. */
int dmd_rew_end_backward(dmd_rew_end* h, int b, int t, const float* g_logits_rew, const float* g_logits_end, float* grads,
                         long long grads_numel, void* workspace, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DIAMOND_B200_H_ */
