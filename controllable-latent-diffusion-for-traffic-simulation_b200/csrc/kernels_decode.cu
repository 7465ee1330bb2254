// VAE LSTM decoder + action de-scaling + unicycle rollout in one kernel, and the indicator kernel.
//   Decoder.forward                         reference models/vae/lstm_vae.py:44-52
//   convert_action_to_state_and_action      reference models/vae/vae_model.py:100-129,157-173
//   unicyle_forward_dynamics('parallel')    reference src/tbsim/models/diffuser_helpers.py:573-639
//   failure_rate_compute / compute_reward   reference models/rl/criticmodel.py:7-64,114-145
//
// Decoder kernel: one CTA owns RB rows ("scene rows"), thread j owns gate row j of the 4H=256 gate
// pre-activations and keeps its recurrent weight row in registers; the hidden states of the RB rows
// live in shared memory and are read as broadcast float4.  The two LSTM layers run as two passes over
// time (layer-0 hidden sequence staged in shared memory), so the per-step critical path is one
// 64-long dot product + one barrier pair.  The kernel is latency/FMA bound, not HBM bound
// (5.26 MFLOP vs ~2 KB per row).
#include "common.cuh"

namespace cld {

struct DynParams {
  float dt, acce_lo, acce_hi, v_lo, v_hi, max_steer, max_yawvel;
  float a_mean, a_std, w_mean, w_std;   // de-scaling of (acc, yawvel): channels 4,5 of nusc_norm_info
};

static DynParams dyn_of(const CldConfig& c) {
  DynParams d;
  d.dt = c.dt; d.acce_lo = c.acce_lo; d.acce_hi = c.acce_hi; d.v_lo = c.v_lo; d.v_hi = c.v_hi;
  d.max_steer = c.max_steer; d.max_yawvel = c.max_yawvel;
  d.a_mean = c.norm_mean[4]; d.a_std = c.norm_std[4]; d.w_mean = c.norm_mean[5]; d.w_std = c.norm_std[5];
  return d;
}

__device__ __forceinline__ float clipf(float x, float lo, float hi) { return fminf(fmaxf(x, lo), hi); }
__device__ __forceinline__ float sigmoid_f(float x) { return 1.0f / (1.0f + expf(-x)); }

// Sequential closed form of the 'parallel' unicycle integration for one row.
// u: metric actions (acc, yawvel) with stride `us`; out6: [T][os] with (x,y,v,yaw[,acc,yawvel]).
__device__ void unicycle_row(const float* u, int us, bool scaled, const float* curr, int T, const DynParams& d,
                             float* out, int os, bool with_actions) {
  float x = curr[0], y = curr[1], s = curr[2], psi = curr[3];
  float vprev = clipf(s, d.v_lo, d.v_hi);
  for (int k = 0; k < T; ++k) {
    float a_raw = u[k * us + 0], w_raw = u[k * us + 1];
    if (scaled) {
      a_raw = __fadd_rn(__fmul_rn(a_raw, d.a_std), d.a_mean);
      w_raw = __fadd_rn(__fmul_rn(w_raw, d.w_std), d.w_mean);
    }
    float a = clipf(a_raw, d.acce_lo, d.acce_hi);
    s = __fadd_rn(s, __fmul_rn(a, d.dt));
    float vnext = clipf(s, d.v_lo, d.v_hi);
    float vbar = __fmul_rn(0.5f, __fadd_rn(vprev, vnext));
    float ve = fabsf(vprev);
    float yb = fminf(__fmul_rn(d.max_steer, ve), __fdiv_rn(d.max_yawvel, fmaxf(ve, 0.1f)));
    yb = fmaxf(yb, 0.1f);
    float w = clipf(w_raw, -yb, yb);
    x = __fadd_rn(x, __fmul_rn(__fmul_rn(vbar, cosf(psi)), d.dt));
    y = __fadd_rn(y, __fmul_rn(__fmul_rn(vbar, sinf(psi)), d.dt));
    psi = __fadd_rn(psi, __fmul_rn(w, d.dt));
    float* o = out + (size_t)k * os;
    o[0] = x; o[1] = y; o[2] = vnext; o[3] = psi;
    if (with_actions) { o[4] = a_raw; o[5] = w_raw; }
    vprev = vnext;
  }
}

struct DecArgs {
  const float *z, *cond, *curr;
  const float *wih0T, *whh0T, *b0, *wih1T, *whh1T, *b1, *c2hT, *c2h_b, *h2a_w, *h2a_b;
  float *act_out, *traj_out, *stash;
  int R, T, C;
  DynParams dyn;
};

template <int RB, int IN, bool SAVE>
__device__ __forceinline__ void lstm_layer(const float* __restrict__ wihT, const float* __restrict__ whhT,
                                           const float* __restrict__ bias, const float* zs, float* hseq,
                                           float* gates, float* hcur, float* stash, int row0, int R, int T) {
  constexpr int H = 64, PPT = RB * H / 256;
  const int j = threadIdx.x;
  float whh[H], wih[IN];
#pragma unroll
  for (int k = 0; k < H; ++k) whh[k] = whhT[k * 256 + j];
#pragma unroll
  for (int k = 0; k < IN; ++k) wih[k] = wihT[k * 256 + j];
  const float bj = bias[j];
  float creg[PPT];
#pragma unroll
  for (int i = 0; i < PPT; ++i) creg[i] = 0.f;
  for (int t = 0; t < T; ++t) {
    float acc[RB];
#pragma unroll
    for (int b = 0; b < RB; ++b) acc[b] = bj;
    if constexpr (IN == 4) {
#pragma unroll
      for (int b = 0; b < RB; ++b) {
        float4 zv = *reinterpret_cast<const float4*>(zs + ((size_t)b * T + t) * 4);
        acc[b] = fmaf(wih[0], zv.x, acc[b]); acc[b] = fmaf(wih[1], zv.y, acc[b]);
        acc[b] = fmaf(wih[2], zv.z, acc[b]); acc[b] = fmaf(wih[3], zv.w, acc[b]);
      }
    } else {
      const float* hin = hseq + (size_t)t * RB * H;
#pragma unroll
      for (int k4 = 0; k4 < IN / 4; ++k4) {
#pragma unroll
        for (int b = 0; b < RB; ++b) {
          float4 hv = *reinterpret_cast<const float4*>(hin + b * H + k4 * 4);
          acc[b] = fmaf(wih[k4 * 4 + 0], hv.x, acc[b]); acc[b] = fmaf(wih[k4 * 4 + 1], hv.y, acc[b]);
          acc[b] = fmaf(wih[k4 * 4 + 2], hv.z, acc[b]); acc[b] = fmaf(wih[k4 * 4 + 3], hv.w, acc[b]);
        }
      }
    }
#pragma unroll
    for (int k4 = 0; k4 < H / 4; ++k4) {
#pragma unroll
      for (int b = 0; b < RB; ++b) {
        float4 hv = *reinterpret_cast<const float4*>(hcur + b * H + k4 * 4);
        acc[b] = fmaf(whh[k4 * 4 + 0], hv.x, acc[b]); acc[b] = fmaf(whh[k4 * 4 + 1], hv.y, acc[b]);
        acc[b] = fmaf(whh[k4 * 4 + 2], hv.z, acc[b]); acc[b] = fmaf(whh[k4 * 4 + 3], hv.w, acc[b]);
      }
    }
#pragma unroll
    for (int b = 0; b < RB; ++b) gates[b * 256 + j] = acc[b];
    __syncthreads();
#pragma unroll
    for (int i = 0; i < PPT; ++i) {
      int p = threadIdx.x + i * 256, b = p >> 6, u = p & 63;
      const float* gr = gates + b * 256;
      float ig = sigmoid_f(gr[u]), fg = sigmoid_f(gr[64 + u]), gg = tanhf(gr[128 + u]), og = sigmoid_f(gr[192 + u]);
      float c = fg * creg[i] + ig * gg;
      creg[i] = c;
      float hv = og * tanhf(c);
      hcur[b * H + u] = hv;
      hseq[((size_t)t * RB + b) * H + u] = hv;
      if (SAVE && row0 + b < R) {
        float* st = stash + ((size_t)t * R + row0 + b) * (5 * H) + u;
        st[0] = ig; st[H] = fg; st[2 * H] = gg; st[3 * H] = og; st[4 * H] = c;
      }
    }
    __syncthreads();
  }
}

template <int RB, bool SAVE>
__global__ void __launch_bounds__(256, 1) lstm_decode_rollout_kernel(DecArgs a) {
  constexpr int H = 64;
  extern __shared__ __align__(16) float smem[];
  const int T = a.T;
  float* zs = smem;                          // [RB][T][4]
  float* hseq = zs + RB * T * 4;             // [T][RB][H]
  float* gates = hseq + (size_t)T * RB * H;  // [RB][256]   (also stages the cond tile)
  float* hcur = gates + RB * 256;            // [RB][H]
  float* h0s = hcur + RB * H;                // [RB][H]
  float* acts = h0s + RB * H;                // [RB][T][2]
  float* trs = acts + RB * T * 2;            // [RB][T][6]
  const int tid = threadIdx.x, row0 = blockIdx.x * RB;

  for (int i = tid; i < RB * T; i += 256) {
    int b = i / T, r = row0 + b;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < a.R) v = reinterpret_cast<const float4*>(a.z)[(size_t)r * T + (i - b * T)];
    reinterpret_cast<float4*>(zs)[i] = v;
  }
  for (int i = tid; i < RB * a.C; i += 256) {
    int b = i / a.C, r = row0 + b;
    gates[i] = (r < a.R) ? a.cond[(size_t)r * a.C + (i - b * a.C)] : 0.f;
  }
  __syncthreads();
  // h0 = cond2hidden(cond) for both layers (lstm_vae.py:46-47); c0 = 0
  for (int p = tid; p < RB * H; p += 256) {
    int b = p >> 6, u = p & 63;
    float acc = a.c2h_b[u];
    for (int k = 0; k < a.C; ++k) acc = fmaf(a.c2hT[k * H + u], gates[b * a.C + k], acc);
    h0s[p] = acc; hcur[p] = acc;
  }
  __syncthreads();
  lstm_layer<RB, 4, SAVE>(a.wih0T, a.whh0T, a.b0, zs, hseq, gates, hcur, a.stash, row0, a.R, T);
  for (int p = tid; p < RB * H; p += 256) hcur[p] = h0s[p];
  __syncthreads();
  lstm_layer<RB, 64, SAVE>(a.wih1T, a.whh1T, a.b1, zs, hseq, gates, hcur,
                           SAVE ? a.stash + (size_t)T * a.R * 5 * H : nullptr, row0, a.R, T);
  // hid2act: one warp per (row, step)
  {
    const int warp = tid >> 5, lane = tid & 31;
    const float w00 = a.h2a_w[lane], w01 = a.h2a_w[lane + 32], w10 = a.h2a_w[H + lane], w11 = a.h2a_w[H + lane + 32];
    for (int it = warp; it < RB * T; it += 8) {
      int b = it / T, t = it - b * T;
      const float* hv = hseq + ((size_t)t * RB + b) * H;
      float h_lo = hv[lane], h_hi = hv[lane + 32];
      float s0 = fmaf(w01, h_hi, w00 * h_lo), s1 = fmaf(w11, h_hi, w10 * h_lo);
#pragma unroll
      for (int o = 16; o; o >>= 1) {
        s0 += __shfl_xor_sync(0xffffffffu, s0, o);
        s1 += __shfl_xor_sync(0xffffffffu, s1, o);
      }
      if (lane == 0) {
        acts[(b * T + t) * 2 + 0] = s0 + a.h2a_b[0];
        acts[(b * T + t) * 2 + 1] = s1 + a.h2a_b[1];
      }
    }
  }
  __syncthreads();
  if (tid < RB && row0 + tid < a.R) {
    float cs[4];
    for (int i = 0; i < 4; ++i) cs[i] = a.curr[(size_t)(row0 + tid) * 4 + i];
    unicycle_row(acts + tid * T * 2, 2, true, cs, T, a.dyn, trs + tid * T * 6, 6, true);
  }
  __syncthreads();
  for (int i = tid; i < RB * T * 2; i += 256) {
    int b = i / (T * 2);
    if (a.act_out && row0 + b < a.R) a.act_out[(size_t)row0 * T * 2 + i] = acts[i];
  }
  for (int i = tid; i < RB * T * 6; i += 256) {
    int b = i / (T * 6);
    if (a.traj_out && row0 + b < a.R) a.traj_out[(size_t)row0 * T * 6 + i] = trs[i];
  }
}

template <int RB>
static size_t dec_smem_bytes(int T, int C) {
  size_t f = (size_t)RB * T * 4 + (size_t)T * RB * 64 + (size_t)RB * (256 > C ? 256 : C) + 2 * RB * 64 +
             (size_t)RB * T * 2 + (size_t)RB * T * 6;
  return f * sizeof(float);
}

template <int RB, bool SAVE>
static int launch_dec(CldHandle* h, const DecArgs& a, cudaStream_t s) {
  size_t smem = dec_smem_bytes<RB>(a.T, a.C);
  auto kern = lstm_decode_rollout_kernel<RB, SAVE>;
  CLD_CUDA_OK(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<(a.R + RB - 1) / RB, 256, smem, s>>>(a);
  CLD_LAUNCH_OK(h, "lstm_decode_rollout_kernel");
  return 0;
}

int decode_rollout(CldHandle* h, const float* z, const float* cond, const float* curr, float* act_out,
                   float* traj_out, bool save, int R, cudaStream_t s) {
  int rc;
  if ((rc = decode_h0(h, cond, h->ws_h0, R, s))) return rc;
  return decode_rollout_h0(h, z, h->ws_h0, curr, act_out ? act_out : h->ws_act, traj_out, save, R, s);
}

__global__ void unicycle_kernel(const float* __restrict__ curr, const float* __restrict__ u, float* __restrict__ out,
                                int R, int T, DynParams d) {
  int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  float cs[4];
  for (int i = 0; i < 4; ++i) cs[i] = curr[(size_t)r * 4 + i];
  unicycle_row(u + (size_t)r * T * 2, 2, false, cs, T, d, out + (size_t)r * T * 4, 4, false);
}

int unicycle(CldHandle* h, const float* curr, const float* u, float* state_out, int R, cudaStream_t s) {
  unicycle_kernel<<<(R + 63) / 64, 64, 0, s>>>(curr, u, state_out, R, h->cfg.horizon, dyn_of(h->cfg));
  CLD_LAUNCH_OK(h, "unicycle_kernel");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Indicators: one warp per row, lanes over time steps; integer results are exact.
// ------------------------------------------------------------------------------------------------
struct IndArgs {
  const float* traj;            // [R,T,6]
  const float* rfa;             // [B,3,3]
  const uint8_t* dmap; int H, W, packed;
  const float* others; const uint8_t* avail; int So;
  uint8_t* offroad; float* coll; float* reward;
  int R, T, N;
  float a_mean, a_std, dt;
};

__global__ void __launch_bounds__(256) indicators_kernel(IndArgs a) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= a.R) return;
  const int ag = row / a.N;
  const float* M = a.rfa + (size_t)ag * 9;
  const float m00 = M[0], m01 = M[1], m02 = M[2], m10 = M[3], m11 = M[4], m12 = M[5];
  const float* tr = a.traj + (size_t)row * a.T * 6;
  int n_off = 0, n_col = 0;
  float jerk = 0.f;
  for (int t = lane; t < a.T; t += 32) {
    const float2 pxy = *reinterpret_cast<const float2*>(tr + t * 6);
    const float px = pxy.x, py = pxy.y;
    // criticmodel.py:101-112: bmm(points, M^T[:2,:2]) + M^T[-1,:2]; then round().long(), clamp
    float xr = __fadd_rn(__fadd_rn(__fmul_rn(px, m00), __fmul_rn(py, m01)), m02);
    float yr = __fadd_rn(__fadd_rn(__fmul_rn(px, m10), __fmul_rn(py, m11)), m12);
    long long ci = llrintf(xr), ri = llrintf(yr);
    if (!(xr == xr)) ci = 0;
    if (!(yr == yr)) ri = 0;
    ci = ci < 0 ? 0 : (ci > a.W - 1 ? a.W - 1 : ci);
    ri = ri < 0 ? 0 : (ri > a.H - 1 ? a.H - 1 : ri);
    const int wb = a.packed ? (a.W + 7) >> 3 : a.W;
    uint8_t dv = a.packed ? (a.dmap[((size_t)ag * a.H + ri) * wb + (ci >> 3)] >> (ci & 7)) & 1 : a.dmap[((size_t)ag * a.H + ri) * wb + ci];
    uint8_t off = dv ? 0 : 1;
    if (a.offroad) a.offroad[(size_t)row * a.T + t] = off;
    n_off += off;
    if (a.others) {
      // four neighbours per iteration, positions fetched whether available or not: eight independent loads in flight per lane
      // instead of a dependent (flag -> position) chain per neighbour
      const float2* oth2 = reinterpret_cast<const float2*>(a.others);
      for (int s = 0; s < a.So; s += 4) {
        uint8_t av[4];
        float2 q[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int sj = s + j < a.So ? s + j : a.So - 1;
          const size_t o = ((size_t)ag * a.So + sj) * a.T + t;
          av[j] = s + j < a.So ? a.avail[o] : (uint8_t)0;
          q[j] = oth2[o];
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float dx = px - q[j].x, dy = py - q[j].y;
          const float d = sqrtf(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
          n_col += (av[j] && d < 0.8f) ? 1 : 0;
        }
      }
    }
    if (t + 1 < a.T) {
      float a0 = (tr[t * 6 + 4] - a.a_mean) / a.a_std, a1 = (tr[(t + 1) * 6 + 4] - a.a_mean) / a.a_std;
      jerk += fabsf((a1 - a0) / a.dt);
    }
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    n_off += __shfl_xor_sync(0xffffffffu, n_off, o);
    n_col += __shfl_xor_sync(0xffffffffu, n_col, o);
    jerk += __shfl_xor_sync(0xffffffffu, jerk, o);
  }
  if (lane == 0) {
    if (a.coll) a.coll[row] = (float)n_col;
    if (a.reward) a.reward[row] = -(float)n_off - (float)n_col - 0.1f * (jerk / (float)(a.T - 1));
  }
}

int indicators(CldHandle* h, const float* traj, const CldScene* sc, uint8_t* offroad, float* coll, float* reward,
               int R, cudaStream_t s) {
  if (!sc || !sc->raster_from_agent || !sc->drivable_map) return fail(h, CLD_ERR_ARG, "scene tensors missing");
  if (sc->num_samp < 1 || R != scene_agents(sc) * sc->num_samp)
    return fail(h, CLD_ERR_ARG, "R=%d does not match %d agents x N=%d", R, scene_agents(sc), sc->num_samp);
  IndArgs a;
  a.traj = traj; a.rfa = sc->raster_from_agent; a.dmap = sc->drivable_map; a.H = sc->map_h; a.W = sc->map_w; a.packed = sc->map_packed;
  a.others = sc->others_pos; a.avail = sc->others_avail; a.So = sc->num_others;
  if (!a.avail) a.others = nullptr;
  a.offroad = offroad; a.coll = coll; a.reward = reward; a.R = R; a.T = h->cfg.horizon; a.N = sc->num_samp;
  a.a_mean = h->cfg.norm_mean[4]; a.a_std = h->cfg.norm_std[4]; a.dt = h->cfg.dt;
  indicators_kernel<<<(R + 7) / 8, 256, 0, s>>>(a);
  CLD_LAUNCH_OK(h, "indicators_kernel");
  return 0;
}

}  // namespace cld
