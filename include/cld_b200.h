/*
 * cld_b200.h -- C ABI of libcld_b200.so: the B200 (sm_100a) implementation of CLD's guided
 * latent-diffusion SAMPLING path.
 *
 * The reference (RoboSafe-Lab/Controllable-Latent-Diffusion-for-Traffic-Simulation) is pure
 * Python/PyTorch and has no FFI; each entry point below names the reference function it replaces
 * (paths relative to the reference root).  INTEGRATION.md shows the ctypes binding a reference
 * maintainer would add to models/dm/dm_model.py.
 *
 * Conventions
 *   - plain pointers and sizes only; every data pointer is a DEVICE pointer owned by the caller
 *     (e.g. torch.Tensor.data_ptr()), contiguous, fp32 unless stated -- except the HOST arrays of
 *     cld_set_schedule and CldScene.scene_start_host;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued asynchronously on it, no
 *     implicit synchronisation, no allocation in the step path (CUDA-graph capturable);
 *   - return 0 on success, a negative CldStatus otherwise; cld_last_error() gives the message;
 *   - a handle belongs to one device and is not thread-safe;
 *   - there is NO CPU fallback and no other-architecture dispatch: cld_create fails on a device
 *     that is not compute capability 10.x.
 *   - row layout: R = S*A*N rows, row = (scene*A + agent)*N + sample  (the reference's
 *     TensorUtils.join_dimensions of [B,N,...], models/dm/dm_model.py:110); ragged scenes
 *     (CldScene.scene_start): R = B*N, row = (scene_start[scene] + agent)*N + sample.
 */
#ifndef CLD_B200_H_
#define CLD_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CldHandle CldHandle;

typedef enum {
  CLD_OK = 0,
  CLD_ERR_ARG = -1,        /* bad argument / shape */
  CLD_ERR_ARCH = -2,       /* device is not sm_100 */
  CLD_ERR_CUDA = -3,       /* CUDA runtime error (message in cld_last_error) */
  CLD_ERR_STATE = -4,      /* weights / schedule not loaded */
  CLD_ERR_UNSUPPORTED = -5 /* configuration outside what the kernels implement */
} CldStatus;

enum { CLD_PREC_FP32 = 0, CLD_PREC_BF16 = 1 };   /* denoiser arithmetic: fp32 SIMT | bf16 tcgen05 */
enum { CLD_SAMPLER_DDPM = 0, CLD_SAMPLER_DDIM = 1 };
enum { CLD_OPT_ADAM = 0, CLD_OPT_SGD = 1 };

/* Mirrors the algo_config keys the reference's hot path reads (SURVEY.md sec. 5 "Config/flags"). */
typedef struct {
  int32_t horizon;          /* algo.horizon (T, multiple of 4)                                   */
  int32_t latent_dim;       /* algo.vae.latent_size (4)                                          */
  int32_t cond_dim;         /* algo.cond_feat_dim (256)                                          */
  int32_t base_dim;         /* algo.base_dim (32): time-embedding width                          */
  int32_t dims[3];          /* base_dim * dim_mults = (64,128,256)                               */
  int32_t hidden;           /* algo.vae.hidden_size (64)                                         */
  int32_t n_timesteps;      /* DmModel(n_timesteps)                                              */
  int32_t max_rows;         /* workspace is sized for this many rows per call                    */
  int32_t precision;        /* CLD_PREC_*                                                        */
  float dt;                 /* algo.step_time (0.1)                                              */
  float acce_lo, acce_hi;   /* algo.dynamics.acce_bound                                          */
  float v_lo, v_hi;         /* Unicycle.vbound default [-10,30] (src/tbsim/dynamics/unicycle.py:9) */
  float max_steer;          /* algo.dynamics.max_steer                                           */
  float max_yawvel;         /* algo.dynamics.max_yawvel                                          */
  float norm_mean[6];       /* algo.nusc_norm_info.diffuser[0]                                   */
  float norm_std[6];        /* algo.nusc_norm_info.diffuser[1]                                   */
} CldConfig;

/* Guidance terms (src/tbsim/utils/guidance_loss.py; defaults src/tbsim/configs/scene_edit_config.py:73-92,302-325). */
typedef struct {
  float w_agent_collision;  /* 50.0 ; 0 disables the term                                        */
  float w_map_collision;    /* 1.0                                                               */
  float w_target_pos;       /* 0.0                                                               */
  int32_t num_disks;        /* 2  (<= 5)                                                         */
  float buffer_dist;        /* 0.2                                                               */
  float decay_rate;         /* 0.9                                                               */
  int32_t num_points_l;     /* 10                                                                */
  int32_t num_points_w;     /* 10                                                                */
  float speed_th;           /* 0.5 (guide_moving_speed_th)                                       */
  float min_target_time;    /* 0.0                                                               */
  int32_t optimizer;        /* CLD_OPT_ADAM                                                      */
  float lr;                 /* 0.3                                                               */
  /* further analytic terms (SURVEY.md sec. 8 f-4); weight 0 disables a term */
  float w_target_speed;     /* TargetSpeedLoss  guidance_loss.py:219-254: mean_t |v_t - v*_t|, v* = CldScene.target_speed */
  float w_acc_limit;        /* AccLimitLoss     guidance_loss.py:1444-1468: mean_t max(|acc_t| - acc_limit, 0)            */
  float acc_limit;
  float w_speed_limit;      /* SpeedLimitLoss   guidance_loss.py:1509-1538: mean_t max(|v_t| - speed_limit, 0)            */
  float speed_limit;
  float w_waypoint;         /* waypoint terms selected per agent by CldScene.wp_mode (TargetPosAtTimeLoss guidance_loss.py:630-670; the
                               branches of GlobalTargetPosAtTimeLoss :930-1031 / GlobalTargetPosLoss :1033-1135, compute_progress_loss :876-927) */
  int32_t grad_steps;       /* optimizer iterations per guided step (perturb's grad_steps); 0 and 1 both mean one, < 0 is CLD_ERR_ARG */
} CldGuidanceConfig;

/* Per-agent scene tensors (the reference's data_batch entries), B = S*A agent rows (ragged: scene_start[S]), scene-major. */
typedef struct {
  int32_t num_scenes;               /* S */
  int32_t agents_per_scene;         /* A >= 1 (ignored with scene_start); any size is guided: one scene's A*N rows must fit CldConfig.max_rows */
  int32_t num_samp;                 /* N */
  const float* extent;              /* [B,3]  data_batch['extent']                               */
  const float* world_from_agent;    /* [B,3,3]                                                   */
  const float* raster_from_agent;   /* [B,3,3]                                                   */
  const float* curr_speed;          /* [B]                                                       */
  const uint8_t* drivable_map;      /* [B,H,W] bool as bytes                                     */
  int32_t map_h, map_w;
  const float* target_pos;          /* [B,2] or NULL                                             */
  const float* others_pos;          /* [B,So,T,2] all_other_agents_future_positions or NULL      */
  const uint8_t* others_avail;      /* [B,So,T]   all_other_agents_future_availability or NULL   */
  int32_t num_others;               /* So */
  int32_t map_packed;               /* 0: drivable_map is [B,H,W] bytes; 1: bit-packed [B,H,(W+7)/8] bytes, pixel x = bit (x & 7) of
                                       byte x >> 3 (numpy.packbits(..., bitorder="little")): 8x fewer bytes to ship per scene      */
  const float* target_speed;        /* [B,T] target speed of every step (TargetSpeedLoss) or NULL */
  /* waypoint guidance (w_waypoint != 0), per agent; the host decides the branch (cld_b200.waypoints mirrors the reference's forward()):
   *   wp_mode 0 none | 1 ||p[wp_time] - g|| | 2 relu(||p[T-1] - g|| - wp_dist) | 3 relu(wp_dist - (||p[0] - g|| - ||p[T-1] - g||)) |
   *           4 TargetPosLoss(g);   g = wp_target in the AGENT frame;   wp_weight = multiplier (A / guided agents of the scene) or NULL */
  const float* wp_target;           /* [B,2] or NULL */
  const int32_t* wp_mode;           /* [B]   or NULL */
  const int32_t* wp_time;           /* [B]   or NULL */
  const float* wp_dist;             /* [B]   or NULL */
  const float* wp_weight;           /* [B]   or NULL */
  /* ragged batches: NULL = every scene holds agents_per_scene agents; otherwise agents_per_scene is ignored and scene s holds agent rows
   * [scene_start[s], scene_start[s+1]): S+1 ascending int32 offsets, [0] = 0, [S] = B, every scene >= 1 agent.
   * Given twice: on the DEVICE for the kernels, and on the HOST for validation, chunking and launch geometry (read during the call only).
   * scene_start_host is the one HOST pointer of this struct, an exception to the device-pointer convention above.
   * cld_sample, cld_guidance_step and cld_indicators take ragged scenes; each scene is guided as if it were alone in the call. */
  const int32_t* scene_start;
  const int32_t* scene_start_host;
} CldScene;

int cld_version(void);
int cld_create(const CldConfig* cfg, CldHandle** out);
void cld_destroy(CldHandle* h);
const char* cld_last_error(const CldHandle* h);   /* h may be NULL: last create() error */

/* Denoiser weights: the 148 tensors of DmModel.model.state_dict() in state-dict order
 * (SURVEY.md sec. 8b), fp32 device pointers; numels[i] (optional, may be NULL) is checked against
 * the element count the layout expects.  Packs them into the kernels' layouts.  On an fp32 handle every call, the first
 * included, is ONE kernel launch with no allocation and no synchronise, so it may be captured in a CUDA graph.  An argument
 * error is reported before anything is written: the loaded weights are unchanged.
 * Replaces: TemporalMapUnet.__init__/load_state_dict (src/tbsim/models/temporal.py:49-120). */
int cld_load_unet(CldHandle* h, const float* const* dev_ptrs, const int64_t* numels, int n, void* stream);

/* LSTM decoder weights, fp32 device pointers in this order:
 * lstm.weight_ih_l0, lstm.weight_hh_l0, lstm.bias_ih_l0, lstm.bias_hh_l0,
 * lstm.weight_ih_l1, lstm.weight_hh_l1, lstm.bias_ih_l1, lstm.bias_hh_l1,
 * cond2hidden.weight, cond2hidden.bias, hid2act.weight, hid2act.bias
 * Replaces: Decoder.__init__ (models/vae/lstm_vae.py:28-43). */
int cld_load_decoder(CldHandle* h, const float* const* dev_ptrs, int n, void* stream);

/* Schedule buffers (HOST fp32 arrays of length n_timesteps), computed by the caller exactly as the
 * reference registers them (models/dm/dm_model.py:29-56). */
int cld_set_schedule(CldHandle* h, const float* x_t_cof, const float* noise_cof,
                     const float* posterior_log_variance_clipped,
                     const float* sqrt_recip_alphas_cumprod, const float* sqrt_recipm1_alphas_cumprod,
                     const float* sqrt_alphas_cumprod, const float* sqrt_one_minus_alphas_cumprod,
                     int n);

/* eps = TemporalMapUnet.forward(x, {'cond_feat': cond}, t)   (src/tbsim/models/temporal.py:122-180)
 * x [R,T,D], cond [R,C], t [R] int64, eps_out [R,T,D]. */
int cld_unet_forward(CldHandle* h, const float* x, const float* cond, const int64_t* t,
                     float* eps_out, int R, void* stream);

/* ---- SURVEY.md sec. 8 f-2: the PPO inner loop's denoiser update ----------------------------------------------------
 * Replaces, for `loss.backward(); opt.step()` of GuideDMLightningModule.ppo_update (src/trainers/guide_dm_trainer.py:127-183):
 * autograd through TemporalMapUnet (src/tbsim/models/temporal.py:122-180), DmModel.log_prob (models/dm/dm_model.py:165-174),
 * the clipped surrogate (guide_dm_trainer.py:158-168) and torch.optim.Adam (guide_dm_trainer.py:59-65).  fp32.
 *
 * cld_unet_train_forward: same result as cld_unet_forward on the fp32 kernels, and keeps every activation the backward needs
 *   in the handle (about 0.85 MB per row; allocated on first use, grows with R).
 * cld_unet_backward: d_eps [R,T,D] = d(loss)/d(eps) -> the gradients of the 148 parameter tensors, WRITTEN (not accumulated) to
 *   grads[i] in state-dict order and layout (Conv1d [cout][cin][k], ConvTranspose1d [cin][cout][k], Linear [out][in]);
 *   dx_out [R,T,D] = d(loss)/d(x) or NULL.  Must directly follow the cld_unet_train_forward of the same rows (no other denoiser
 *   call on this handle in between).  No atomics: a step is bit-reproducible. */
int cld_unet_train_forward(CldHandle* h, const float* x, const float* cond, const int64_t* t, float* eps_out, int R, void* stream);
int cld_unet_backward(CldHandle* h, const float* d_eps, float* const* grads, int n, float* dx_out, int R, void* stream);

/* PPO head: logp_new[r] = mean_{T,D} Normal(x_t_cof[t] x_t - noise_cof[t] eps, exp(.5 logvar[t])).log_prob(x_tm1),
 * loss = -(1/R) sum_r min(ratio A, clamp(ratio, 1-clip, 1+clip) A), ratio = exp(logp_new - logp_old), A = reward - baseline;
 * d_eps_out [R,T,D] = d(loss)/d(eps).  logp_new_out [R], loss_out [1], d_eps_out may be NULL.  baseline_dev (may be NULL): the baseline
 * as ONE device float, read by the kernel instead of `baseline` -- for callers that replay the update as a CUDA graph. */
int cld_ppo_head(CldHandle* h, const float* eps, const float* x_t, const float* x_tm1, const int64_t* t, const float* logp_old,
                 const float* reward, float baseline, const float* baseline_dev, float clip_eps, float* logp_new_out, float* loss_out,
                 float* d_eps_out, int R, void* stream);
/* F.mse_loss(noise, eps) of DmModel.compute_losses (models/dm/dm_model.py:83-90) and its gradient d_eps_out (may be NULL). */
int cld_mse_head(CldHandle* h, const float* eps, const float* noise, float* loss_out, float* d_eps_out, int R, void* stream);
/* forward + PPO head + backward in one call (the body of one minibatch iteration of ppo_update up to `opt.step()`). */
int cld_ppo_grad(CldHandle* h, const float* x_t, const float* x_tm1, const float* cond, const int64_t* t, const float* logp_old,
                 const float* reward, float baseline, const float* baseline_dev, float clip_eps, float* const* grads, int n,
                 float* logp_new_out, float* loss_out, int R, void* stream);
/* The same step with the step counter (int64, incremented by the call) and the learning rate (double) in DEVICE memory, so that a
 * captured CUDA graph of the whole update (cld_ppo_grad + this + cld_load_unet on the loaded handle) can be replayed: no host-side
 * scalar changes between replays. */
int cld_adam_step_dev(CldHandle* h, float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t numel, const double* lr_dev,
                      int64_t* step_dev, double beta1, double beta2, double eps, double weight_decay, void* stream);
/* tf32 != 0: the stride-1 convolutions of the training step (forward and data gradient) run on the tensor pipe (tcgen05 kind::tf32,
 * fp32 operands read with 10 mantissa bits, fp32 accumulation); 0 (default): everything in fp32 on the CUDA cores (1e-4 parity mode). */
int cld_train_set_precision(CldHandle* h, int tf32);
/* torch.optim.Adam step (amsgrad off; weight_decay added to the gradient) on ONE flat fp32 vector of `numel` elements; `step`
 * counts from 1; the hyper-parameters are doubles because torch derives its scalar factors (1 - beta, bias corrections) in double.
 * The caller keeps the parameters of the model as views of that vector. */
int cld_adam_step(CldHandle* h, float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t numel, double lr,
                  double beta1, double beta2, double eps, double weight_decay, int step, void* stream);

/* Debug/verification hook: registers a tap; the NEXT cld_unet_forward calls copy the channels-last
 * activation [R,T',C] produced by stage `stage_index` (0..16: downs.0.0, downs.0.1, downs.0.2, ...,
 * mid_block1, mid_block2, ups.0.0, ..., ups.1.2, final_conv.0) into `out` (fp32).  out == NULL
 * removes the tap.  Returns elements per row of that stage (negative on error). */
int cld_unet_debug_stage(CldHandle* h, int stage_index, float* out, int R, void* stream);

/* One posterior step (models/dm/dm_model.py:144-163):
 *   DDPM: mean = x_t_cof[t]*x - noise_cof[t]*eps ; x' = mean + 1[t!=0]*exp(.5*logvar[t])*noise
 *   DDIM (eta=0, t_next<0 means final): x0 = sqrt_recip[t]*x - sqrt_recipm1[t]*eps ;
 *         x' = mean = sqrt_acp[t_next]*x0 + sqrt(1-acp[t_next])*eps
 * noise may be NULL (treated as 0).  mean_out may be NULL.  x_out may alias x. */
int cld_posterior_step(CldHandle* h, const float* x, const float* eps, const float* noise,
                       int t, int t_next, int sampler, float* x_out, float* mean_out, int R,
                       void* stream);

/* x' = mean + 1[t!=0]*sigma[t]*noise (the noise injection applied after guidance). */
int cld_add_noise(CldHandle* h, const float* mean, const float* noise, int t, float* x_out, int R,
                  void* stream);

/* act = Decoder.forward(z, cond) (models/vae/lstm_vae.py:44-52) fused with
 * VaeModel.convert_action_to_state_and_action(act, curr, descaled_output=True)
 * (models/vae/vae_model.py:100-129; unicycle: src/tbsim/models/diffuser_helpers.py:573-639).
 * z [R,T,4], cond [R,C], curr [R,4] -> act_out [R,T,2] scaled actions (may be NULL),
 * traj_out [R,T,6] metric (x,y,v,yaw,acc,yawvel). */
int cld_decode_rollout(CldHandle* h, const float* z, const float* cond, const float* curr,
                       float* act_out, float* traj_out, int R, void* stream);

/* Unicycle rollout alone (diffuser_helpers.py:573-639): u [R,T,2] metric actions -> [R,T,4]. */
int cld_unicycle(CldHandle* h, const float* curr, const float* u, float* state_out, int R,
                 void* stream);

/* failure_rate_compute / compute_reward indicators (models/rl/criticmodel.py:7-64,114-145).
 * traj [R,T,6] metric, rows map to agents by row / num_samp.
 * offroad_out [R,T] bytes (1 = off the drivable area), coll_out [R] fp32 collision counts,
 * reward_out [R] fp32 (may be NULL). */
int cld_indicators(CldHandle* h, const float* traj, const CldScene* scene, uint8_t* offroad_out,
                   float* coll_out, float* reward_out, int R, void* stream);

/* PerturbationGuidance.perturb (guidance_loss.py:2221-2282) with decoder = lstm_dec and
 * transform = convert_action_to_state_and_action, one scene per reference call: g->grad_steps
 * iterations of  g = dL/dz (analytic backward), then one step of a fresh torch.optim.Adam
 * (step 1: z - lr*g/(|g|+1e-8)) or SGD (z - lr*g).  Iteration 1 reads z_mean, later ones the
 * previous iteration's z; the Adam moments of a multi-step call live in the handle ([max_rows,T,4]
 * x 2, allocated by the first call with grad_steps > 1).  cond/curr are per ROW ([R,C], [R,4]).
 * grad_out [R,T,4] and loss_out [7,R] (agent_collision, map_collision, target_pos, target_speed,
 * acc_limit, speed_limit, waypoint per row) may be NULL; with grad_steps > 1 they hold the gradient
 * and the losses of the LAST iteration, as perturb returns them.  z_out may alias z_mean. */
int cld_guidance_step(CldHandle* h, const float* z_mean, const float* cond, const float* curr,
                      const CldScene* scene, const CldGuidanceConfig* g, float* z_out,
                      float* grad_out, float* loss_out, int R, void* stream);

/* Whole sampler: DmModel.sample_traj (models/dm/dm_model.py:103-142) + optional guidance
 * (template src/tbsim/models/diffuser.py:843-929) + decode/rollout + indicators.
 *   x_init [R,T,D] (NULL with seed!=0: drawn in-kernel); noises [K,R,T,D] or NULL with seed!=0 for in-kernel
 *   Philox4x32-10 noise.  row_offset = GLOBAL id of row 0 of this call (0 for an unsharded call): the Philox
 *   counter of an element is (global row, element, step), so a shard / chunk / lane of a batch draws exactly
 *   what the unsharded batch would (SURVEY.md sec. 8e).
 *   cond [R,C], curr [R,4] per row; scene/g may be NULL (unguided, no indicators).  Every guided
 *   step runs the g->grad_steps iterations of cld_guidance_step on the posterior mean.
 * Outputs (any may be NULL): x0 [R,T,D], x1 [R,T,D] (written only if step index 1 is visited;
 * *x1_valid says so), traj [R,T,6], offroad [R,T], coll [R]. */
int cld_sample(CldHandle* h, const float* x_init, const float* noises, uint64_t seed,
               int64_t row_offset, const float* cond, const float* curr, const CldScene* scene,
               const CldGuidanceConfig* g, int stride, int sampler, float* x0_out, float* x1_out,
               int* x1_valid, float* traj_out, uint8_t* offroad_out, float* coll_out, int R,
               void* stream);

/* Hardware self-test of the tcgen05 building blocks (no handle): stages a 128B-swizzled A image and
 * B image (device pointers) in shared memory, issues nk16 UMMAs (M=128, N, K=16) whose A descriptor starts
 * a_start_off bytes into the image with sbo_a bytes between 8-row groups, returns D [128][N] fp32. */
int cld_tc_selftest(const void* a_img, int a_bytes, const void* b_img, int b_bytes, int a_start_off,
                    int sbo_a, int N, int nk16, int base_offset, float* d_out, void* stream);

/* Measurement hooks (bench.py): number of kernels this handle has launched, and CUDA-event brackets
 * around the phases of cld_sample on the caller's stream (kind 0 denoiser forward, 1 posterior /
 * noise step, 2 guidance step, 3 decode + rollout + indicators).  cld_profile_end synchronises on the
 * last recorded event and returns summed milliseconds and bracket counts per kind. */
unsigned long long cld_launch_count(const CldHandle* h);
int cld_profile_begin(CldHandle* h);
int cld_profile_end(CldHandle* h, double* ms_by_kind, int* count_by_kind, int nkinds);

/* ---------------------------------------------------------------------------------------------
 * Context encoder (SURVEY.md sec. 8 row a14): ContextEncoder.forward (models/context_utils.py:40-61), the provider
 * of cond_feat for the sampler.  Own handle type (its workspace is sized per agent, not per row).
 *   map_encoder  = torchvision ResNet-18, 34-channel 7x7 stem, eval-mode BatchNorm, fc 512 -> 256
 *                  (src/tbsim/models/base_models.py:573-607, src/tbsim/models/diffuser_helpers.py:297-348)
 *   agent_state_encoder / process_cond_mlp = base_models.MLP with LayerNorm (base_models.py:58-66)
 * Arithmetic: bf16 tcgen05 implicit-GEMM convolutions with fp32 accumulation, fp32 BatchNorm / residual / head. */
typedef struct CldContext CldContext;

/* Workspace for up to max_agents agents per forward call (processed in chunks of <= 2048 agents, 6 MB each) on the
 * CURRENT device; fails with CLD_ERR_ARCH on a device that is not compute capability 10.x. */
int cld_context_create(int max_agents, CldContext** out);
void cld_context_destroy(CldContext* c);
const char* cld_context_last_error(const CldContext* c);   /* c may be NULL: last create() error */

/* The 130 fp32 tensors of ContextEncoder.state_dict() in state-dict order WITHOUT the 20 `num_batches_tracked`
 * entries (device pointers; numels optional).  Packs the convolution weights into MMA-ready bf16 tiles and folds the
 * BatchNorm running statistics into a per-channel scale / shift.  Replaces ContextEncoder.__init__/load_state_dict. */
int cld_context_load(CldContext* c, const float* const* dev_ptrs, const int64_t* numels, int n, void* stream);

/* cond_feat [B,256] = ContextEncoder.forward(data_batch)['cond_feat'] for image [B,34,224,224] (NCHW fp32) and
 * curr_states [B,4] = (x, y, vel, yaw) of batch_utils.get_current_states (src/tbsim/utils/batch_utils.py:61-65).
 * map_feat_out (optional) [B,256] receives the ResNet's fc output.  Verification tap: tap_stage 0 (stem + max-pool),
 * 1..4 (layer1..layer4) copies that activation to tap_out as fp32 NCHW (B <= chunk); pass -1 / NULL otherwise. */
int cld_context_forward(CldContext* c, const float* image, const float* curr_states, int B, float* cond_feat,
                        float* map_feat_out, int tap_stage, float* tap_out, void* stream);

/* The same from the UN-RASTERISED inputs of the data layer: rasterize_agents (src/tbsim/utils/trajdata_utils.py:123-156, called
 * by parse_node_centric :395-420) fused with the encoder's raster layout, so the 6.8 MB/agent fp32 image never exists.
 *   maps [B,3,224,224] fp32 map layers; hist_pos [B,A,31,2] fp32 history positions in the ego frame, agent 0 = the ego;
 *   hist_mask [B,A,31] bytes (availability); raster_from_agent [B,3,3] fp32.
 * cond_feat == NULL rasterises only; image_out (optional) [B,34,224,224] fp32 receives the image rasterize_agents returns
 * (history channel t: +1 at the ego's pixel, -1 at the other agents'; then the map layers). */
int cld_context_forward_history(CldContext* c, const float* maps, const float* hist_pos, const uint8_t* hist_mask,
                                const float* raster_from_agent, int num_hist_agents, const float* curr_states, int B,
                                float* cond_feat, float* map_feat_out, float* image_out, void* stream);

unsigned long long cld_context_launch_count(const CldContext* c);
/* 2*MAC per agent of the 20 convolutions as executed (includes the zero-padded K of the stem). */
double cld_context_conv_flops(const CldContext* c);

#ifdef __cplusplus
}
#endif
#endif /* CLD_B200_H_ */
