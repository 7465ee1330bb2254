// Shared declarations of libcld_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>

#include "../../include/cld_b200.h"

#define CLD_MAX_T 128          // horizon upper bound baked into per-thread scan arrays
#define CLD_TB_TOTAL_MAX 4096  // upper bound of the concatenated time-bias width

namespace cld {

// ------------------------------------------------------------------------------------------------
// U-Net plan (src/tbsim/models/temporal.py:49-120): 12 residual blocks, 2 down convs, 2 up convs,
// final block.  Weights are re-packed at load time; fp32 packing: conv taps as [tap][cin][cout].
// ------------------------------------------------------------------------------------------------
struct ConvW {
  float* w = nullptr;   // fp32 [ntaps][cin][cout]
  float* wt = nullptr;  // fp32 [ntaps][cout][cin]: B operand (K-major) of the tensor-core training forward (train_tc.cu)
  float* b = nullptr;   // [cout]
  int cin = 0, cout = 0, ntaps = 0;
};
struct GnW {
  float* g = nullptr;
  float* b = nullptr;
};
struct ResBlockW {
  ConvW c0, c1, res;    // res.w == nullptr -> identity
  GnW n0, n1;
  int tb_off = 0;       // offset of this block's slice inside the concatenated time-bias
  int cin = 0, cout = 0;
};

struct UnetW {
  // time embedding MLP
  float *t1_w = nullptr, *t1_b = nullptr, *t2_w = nullptr, *t2_b = nullptr;   // [4d,d],[4d],[d,4d],[d]
  float* freqs = nullptr;   // [d/2] sinusoid frequencies (diffuser_helpers.py:27-29)
  // concatenated per-block Linear(288->cout): packed [288][tb_total] + bias[tb_total]
  float* tb_w = nullptr;
  float* tb_wt = nullptr;   // the same weights as [tb_total][tdim] (K contiguous): B operand of the tensor-core training forward
  float* tb_b = nullptr;
  int tb_total = 0;
  ResBlockW rb[12];     // downs.0.0 .. ups.1.1 in execution order
  ConvW down[2];        // k3 s2 p1
  ConvW up[2][2];       // transposed conv split in 2 output phases, 2 taps each
  float* up_b[2] = {nullptr, nullptr};
  ConvW fin0;           // final Conv1dBlock conv
  GnW fin0n;
  ConvW fin1;           // 1x1 conv to latent dim
  bool loaded = false;
};

struct DecoderW {
  // transposed copies [in][4H] for the forward kernel (coalesced register loads)
  float *wih0 = nullptr, *whh0 = nullptr, *b0 = nullptr;   // [4,256],[64,256],[256] (b_ih+b_hh)
  float *wih1 = nullptr, *whh1 = nullptr, *b1 = nullptr;   // [64,256],[64,256],[256]
  // original nn.LSTM layouts [4H][in] for the backward kernel
  float *wih0_raw = nullptr, *whh0_raw = nullptr, *wih1_raw = nullptr, *whh1_raw = nullptr;
  float *c2h_w = nullptr, *c2h_b = nullptr;                // transposed [C,64], [64]
  float *h2a_w = nullptr, *h2a_b = nullptr;                // [2,64],[2]
  float *w0p = nullptr, *w1p = nullptr;                    // packed forward weights for kernels_lstm.cu
  float *w1t = nullptr, *w0t = nullptr;                    // packed transposed weights for the backward
  bool loaded = false;
};

struct Schedule {
  std::vector<float> x_t_cof, noise_cof, logvar, sqrt_recip, sqrt_recipm1, sqrt_acp, sqrt_1macp;
  bool loaded = false;
};

}  // namespace cld

namespace cld {
// State-dict layout of the denoiser: the tensors of DmModel.model.state_dict() that cld_load_unet takes and cld_unet_backward writes,
// by index.  Depends on the config only (built at cld_create).
struct BlkIdx { int tw, tb, c0w, c0b, g0, b0, c1w, c1b, g1, b1, rw, rb; };   // rw = rb = -1: identity residual
struct UnetLayout {
  std::vector<int64_t> numel;   // element count of every state-dict tensor
  int tmlp[4];                  // time_mlp: Linear(d, 4d) weight, bias; Linear(4d, d) weight, bias
  BlkIdx blk[12];               // residual blocks in execution order (UnetW::rb)
  int down[2][2], up[2][2];     // {weight, bias} of the down / up convolutions
  int fin[6];                   // final_conv: conv weight, bias, GroupNorm weight, bias; 1x1 conv weight, bias
};

// one entry of the weight pack table: cld_load_unet packs all of them in one launch
struct PackJob {
  int kind;            // 0: conv [cout][cin][K] -> [tap][cin][ld] (+off); 1: -> [tap][cout][cin]; 2: flat copy
  int src;             // index into the state-dict pointer list
  float* dst;
  int cout, cin, K, ntaps, ks[5], ld, off, transposed, total, blk0;
};
}  // namespace cld

struct CldHandle {
  CldConfig cfg;
  int device = 0;
  int num_sms = 0;
  std::string err;
  cld::UnetW unet;
  cld::UnetLayout unet_layout;
  cld::DecoderW dec;
  cld::Schedule sched;
  std::vector<void*> allocs;       // everything cudaMalloc'ed by the handle
  // fp32 denoiser workspace (sized for cfg.max_rows)
  float* act[8] = {nullptr};       // activation buffers, each max_rows * act_elems floats
  size_t act_elems = 0;            // per-row elements of one activation buffer
  float* tcm = nullptr;            // [max_rows, 32+cond] Mish([t_emb, cond])
  float* tbias = nullptr;          // [max_rows, tb_total]
  float* tvec = nullptr;           // [tb_total] per-step time part of the bias (sampler: uniform t)
  float* tvec_all = nullptr;       // [n_timesteps, tb_total]: the same for every timestep, filled once after a weight load (cld_sample)
  bool tvec_all_valid = false;
  cudaEvent_t ev_tvec = nullptr;   // recorded after the table was filled: later calls on another stream wait for it
  cudaStream_t tvec_stream = nullptr;
  // guidance / decode workspace
  float* stash = nullptr;          // LSTM forward stash, see stash_index()
  float* ws_act = nullptr;         // [max_rows, T, 2]
  float* ws_h0 = nullptr;          // [max_rows, H] cond2hidden(cond): LSTM initial state
  float* ws_dh0 = nullptr;         // [T, max_rows, H] d(loss)/d(h0_t) coming down from layer 1 (backward)
  float* ws_traj = nullptr;        // [max_rows, T, 6]
  float* ws_dtraj = nullptr;       // [max_rows, T, 4]
  float* ws_dtraj2 = nullptr;      // [max_rows, T, 4] map-collision part when it runs concurrently (bf16 mode sampler)
  float* ws_dacc = nullptr;        // [max_rows, T] d/d(acc) of the acc-limit guidance term
  // Adam moments (m, v) of a guided step with grad_steps > 1, [max_rows, T, 4] each: allocated on first use
  float* ws_adam_m = nullptr;
  float* ws_adam_v = nullptr;
  // map-collision guidance: work list of the (row, step) items whose footprint may cross a road edge (+ 2 counters), and the
  // one-bit-per-pixel copy of byte-per-pixel drivable maps that the screen reads (guidance_prepare_maps; bit-packed scenes are read in place)
  int* map_work = nullptr;
  uint8_t* map_bits = nullptr;
  size_t map_bits_bytes = 0;
  const void* screen_src = nullptr;        // the drivable_map pointer the screen data belongs to (nullptr: none)
  const uint8_t* screen_pk = nullptr;      // where the screen reads: map_bits or the scene's own packed maps
  int screen_agents = 0, screen_h = 0, screen_w = 0, screen_packed = 0, screen_pitch = 0;
  cudaStream_t aux_stream = nullptr;   // forked from / joined to the caller's stream with the two events below
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  float* ws_loss = nullptr;        // [3, max_rows]
  float* ws_eps = nullptr;         // [max_rows, T, D]
  float* ws_mean = nullptr;        // [max_rows, T, D]
  float* ws_x = nullptr;           // [max_rows, T, D]
  int64_t* ws_t = nullptr;         // [max_rows]
  // debug tap
  int dbg_stage = -1;
  float* dbg_out = nullptr;
  // measurement: kernels launched by this handle; optional CUDA-event brackets around the phases of
  // cld_sample (0 denoiser, 1 posterior/noise, 2 guidance, 3 decode+indicators)
  unsigned long long launches = 0;
  bool profiling = false;
  std::vector<cudaEvent_t> ev_pool;
  std::vector<int> ev_kind;      // kind of bracket i (events 2i, 2i+1)
  size_t ev_used = 0;
  // bf16 tensor-core path (opaque, owned by unet_tc.cu)
  void* tc = nullptr;
  // tensor-core LSTM decoder (opaque, owned by kernels_lstm_tc.cu); used when cfg.precision == CLD_PREC_BF16
  void* lstm_tc = nullptr;
  bool use_lstm_tc = false;
  // denoiser training state (opaque, owned by kernels_unet_train.cu): activation stash + gradient scratch, allocated on first use
  void* train = nullptr;
  unsigned long long sched_version = 0;   // bumped by cld_set_schedule
  // the pack table cld_load_unet launches (device copy, built at cld_create), and the grid it needs
  cld::PackJob* pack_jobs = nullptr;
  int pack_njobs = 0, pack_blocks = 0;
  void* train_tc = nullptr;        // tensor-map cache of the tf32 tensor-core convolutions (train_tc.cu)
  bool train_tf32 = false;         // cld_train_set_precision: stride-1 convolutions of the training step on the tensor pipe
  // debug switches, read from the environment ONCE at cld_create (never inside the step path)
  bool env_train_serial = false;   // CLD_TRAIN_SERIAL=1: parameter gradients on the caller's stream instead of the handle's second stream
  bool env_lstm_bwd_simt = false, env_guidance_nofork = false, env_lstm_prof = false, env_map_stats = false, env_map_exhaustive = false;
  int env_lstm_pf = 3;
};

namespace cld {
// LSTM stash (gate activations i, f, g, o and the cell state c of every step, for the analytic backward):
// [layer][t][row block of 8][value 0..4][unit 0..63][row in block].  A SIMT thread (8 rows x 1 unit) moves 32
// contiguous bytes and a warp of consecutive units 1 KB; a tensor-core epilogue warp (lane = row) touches 4 full
// 32-byte sectors per store.  Rows are padded to a multiple of 64.
__host__ __device__ inline size_t stash_index(int layer, int t, int T, int R, int row, int v, int u) {
  const size_t rblk = (size_t)((R + 63) >> 6) * 8;
  return (((((size_t)layer * T + t) * rblk + (size_t)(row >> 3)) * 5 + v) * 64 + u) * 8 + (row & 7);
}
constexpr int STASH_V_STRIDE = 64 * 8;   // floats between consecutive values v for the same (row block, unit)
int fail(CldHandle* h, int code, const char* fmt, ...);
#define CLD_CUDA_OK(h, expr)                                                                   \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess)                                                                     \
      return cld::fail(h, CLD_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                       __FILE__, __LINE__);                                                    \
  } while (0)
#define CLD_LAUNCH_OK(h, name)                                                             \
  do {                                                                                     \
    cudaError_t _e = cudaGetLastError();                                                   \
    if (_e != cudaSuccess)                                                                 \
      return cld::fail(h, CLD_ERR_CUDA, "launch of %s failed: %s", name, cudaGetErrorString(_e)); \
    if (h) ++(h)->launches;                                                                \
  } while (0)

// event brackets for cld_sample phases (no-ops unless h->profiling)
int prof_begin(CldHandle* h, int kind, cudaStream_t s);
int prof_end(CldHandle* h, cudaStream_t s);
// ---- kernels_unet_fp32.cu
int unet_forward_fp32(CldHandle* h, const float* x, const float* cond, const int64_t* t, float* eps,
                      int R, cudaStream_t s);
int unet_stage_elems(const CldHandle* h, int stage);
int unet_time_bias(CldHandle* h, const float* cond, const int64_t* t, int R, cudaStream_t s);   // per-row t -> h->tcm, h->tbias
int unet_time_cond(CldHandle* h, const float* cond, const int64_t* t, int R, cudaStream_t s);   // only h->tcm = Mish([t_emb, cond])
int unet_cond_bias(CldHandle* h, const float* cond, int R, cudaStream_t s);   // -> h->tbias (cond part + bias)
int unet_time_vec(CldHandle* h, int t, cudaStream_t s);                        // -> h->tvec
int unet_time_vec_to(CldHandle* h, int t, float* dst, cudaStream_t s);
int gn_mish_launch(CldHandle* h, const float* in, const GnW& n, const float* tbias, int tb_stride, const float* res, float* out,
                   int T, int C, int R, cudaStream_t s);
// ---- kernels_unet_train.cu (SURVEY.md sec. 8 f-2)
int unet_train_forward(CldHandle* h, const float* x, const float* cond, const int64_t* t, float* eps, int R, cudaStream_t s);
int unet_train_backward(CldHandle* h, const float* d_eps, float* const* grads, int n, float* dx_out, int R, cudaStream_t s);
int ppo_head(CldHandle* h, const float* eps, const float* x_t, const float* x_tm1, const int64_t* t, const float* logp_old,
             const float* reward, float baseline, const float* baseline_dev, float clip, float* logp_new, float* loss_out, float* d_eps, int R,
             cudaStream_t s);
int adam_step_dev(CldHandle* h, float* p, const float* g, float* m, float* v, size_t n, const double* lr_dev, long long* step_dev, double b1,
                  double b2, double eps, double wd, cudaStream_t s);
int mse_head(CldHandle* h, const float* eps, const float* noise, float* loss_out, float* d_eps, int R, cudaStream_t s);
int adam_step(CldHandle* h, float* p, const float* g, float* m, float* v, size_t n, double lr, double b1, double b2, double eps, double wd,
              int step, cudaStream_t s);
float* train_deps_buffer(CldHandle* h);
// ---- train_tc.cu
bool tfconv_supported(int c0, int c1, int N, int Tp);
int tfconv_launch(CldHandle* h, const float* in0, int c0, const float* in1, int c1, int Ta, int tstride, int Tp, const float* w, int planes,
                  int ntaps, const int* wtap, const int* toff, const float* bias, float* out, int Tout, int ostride, int ooff, int N, int accum,
                  int R, cudaStream_t s);
bool tfwgrad_supported(int c0, int c1, int cout, int Tp, int R);
int tfwgrad_launch(CldHandle* h, const float* in0, int c0, const float* in1, int c1, int Ta, int a_stride, int Tp, const float* dout, int Td,
                   int d_stride, int d_toff, int cout, int ntaps, const int* toff, float* part, size_t part_floats, int max_splits, int R,
                   int* splits_out, cudaStream_t s);
void train_tc_destroy(CldHandle* h);
void train_destroy(CldHandle* h);
void train_invalidate(CldHandle* h);     // the time / cond bias buffers the backward reads were overwritten
// ---- kernels_step.cu
// in-kernel noise: Philox4x32-10(key = seed, counter = (idx_base + element quad, seq)); idx_base = GLOBAL row id * T*D/4 and
// seq = position of the step in the schedule, so the draw of a row does not depend on sharding / chunking / lanes
int posterior_step(CldHandle* h, const float* x, const float* eps, const float* noise, uint64_t seed,
                   uint64_t seq, uint64_t idx_base, int t, int t_next, int sampler, float* x_out, float* mean_out, int R,
                   cudaStream_t s);
int add_noise(CldHandle* h, const float* mean, const float* noise, uint64_t seed, uint64_t seq, uint64_t idx_base, int t,
              float* x_out, int R, cudaStream_t s);
int philox_fill(CldHandle* h, uint64_t seed, uint64_t seq, uint64_t idx_base, float* out, int R, cudaStream_t s);
int fill_t(CldHandle* h, int64_t* t, int value, int R, cudaStream_t s);
// ---- kernels_decode.cu
int decode_rollout(CldHandle* h, const float* z, const float* cond, const float* curr, float* act_out,
                   float* traj_out, bool save, int R, cudaStream_t s);
int unicycle(CldHandle* h, const float* curr, const float* u, float* state_out, int R, cudaStream_t s);
// optimizer iteration `iter` (1-based) of a guided step.  m == nullptr: the single-iteration update (torch's first Adam step, or
// SGD), no moment traffic.  Otherwise Adam with moments m / v [R,T,4]: iteration 1 writes m = 0.1 g, v = 0.001 g^2 next to the
// first-step update, iteration >= 2 reads and updates them and steps z -= step_size * m / (sqrt(v) / bc2_sqrt + 1e-8).
struct GuideOpt {
  int iter = 1;
  float* m = nullptr;
  float* v = nullptr;
  float step_size = 0.f;     // lr / (1 - 0.9^iter)
  float bc2_sqrt = 0.f;      // sqrt(1 - 0.999^iter)
};
// ---- kernels_lstm.cu
int decode_h0(CldHandle* h, const float* cond, float* h0, int R, cudaStream_t s);
int decode_backward_update2(CldHandle* h, const float* z_mean, const float* act, const float* curr, const float* dtraj,
                            const float* dtraj2, const float* dacc, const CldGuidanceConfig* g, const GuideOpt& opt, float* z_out,
                            float* grad_out, int R, cudaStream_t s);
int decode_rollout_h0(CldHandle* h, const float* z, const float* h0, const float* curr, float* act_out, float* traj_out,
                      bool save, int R, cudaStream_t s);
int decode_rollout_h0_tc(CldHandle* h, const float* z, const float* h0, const float* curr, float* act_out, float* traj_out,
                         bool save, int R, cudaStream_t s);
int decode_backward_update_tc(CldHandle* h, const float* z_mean, const float* act, const float* curr, const float* dtraj,
                              const float* dtraj2, const float* dacc, const CldGuidanceConfig* g, const GuideOpt& opt, float* z_out,
                              float* grad_out, int R, cudaStream_t s);
void lstm_tc_destroy(CldHandle* h);
int indicators(CldHandle* h, const float* traj, const CldScene* sc, uint8_t* offroad, float* coll,
               float* reward, int R, cudaStream_t s);
// ---- kernels_guidance.cu
// dtraj_map != nullptr (and loss == nullptr): the map-collision part runs concurrently on the handle's auxiliary stream and
// writes its own buffer; the caller adds the two
// dacc [R,T]: d/d(acc) of the acc-limit term (written when g->w_acc_limit != 0; consumed by the unicycle backward)
int guidance_loss_grad(CldHandle* h, const float* traj, const CldScene* sc, const CldGuidanceConfig* g,
                       float* dtraj, float* dtraj_map, float* dacc, float* loss, int R, cudaStream_t s);
// the screen of the map-collision term reads the drivable maps with one bit per pixel: byte-per-pixel maps are packed here, once per
// cld_sample chunk / cld_guidance_step call (the maps of a call do not change between denoising steps)
int guidance_prepare_maps(CldHandle* h, const CldScene* sc, cudaStream_t s);
int decode_backward_update(CldHandle* h, const float* z_mean, const float* act, const float* curr,
                           const float* dtraj, const CldGuidanceConfig* g, float* z_out, float* grad_out,
                           int R, cudaStream_t s);
}  // namespace cld
