// LSTM decoder forward as a sequence of small register-tiled GEMMs (fp32, packed FFMA2), fused with the
// action de-scaling and the unicycle rollout.
//   Decoder.forward                         reference models/vae/lstm_vae.py:44-52
//   convert_action_to_state_and_action      reference models/vae/vae_model.py:100-129,157-173
//   unicyle_forward_dynamics('parallel')    reference src/tbsim/models/diffuser_helpers.py:573-639
//
// One CTA owns 32 rows.  Both layers' weights live in shared memory (200 KB, packed [k pair][unit][gate][2]) for the
// whole kernel; per time step the gate pre-activations of a layer are a [32 x K] x [K x 256] product.  A thread owns
// ONE hidden unit for 8 rows and all four gates of it (i, f, g, o) in BOTH layers, so the LSTM cell update needs no
// exchange: 32 packed accumulators per thread, the cell states stay in registers for all T steps.  The two layers
// run skewed by one step (iteration i: layer 0 computes step i, layer 1 computes step i - 1; both read h0_{i-1}),
// so a time step costs two block barriers.  With SAVE the gate activations and cell states are stashed for the
// analytic backward (kernels_guidance.cu).
#include <stdlib.h>

#include "common.cuh"
#include "lstm_shared.cuh"

namespace cld {

namespace {
constexpr int LS_RB = 32;        // rows per CTA
constexpr int LS_RP = 34;        // padded row count of the state tiles (bank spread for the unit-major stores)
constexpr int LS_H = 64;
constexpr int LS_KP0 = 34;       // layer 0: (4 inputs + 64 hidden) / 2
constexpr int LS_KP1 = 64;       // layer 1: (64 + 64) / 2
constexpr int LS_THREADS = 256;
// shared memory (floats)
constexpr int LS_W0 = 0;
constexpr int LS_W1 = LS_W0 + LS_KP0 * LS_H * 8;
constexpr int LS_XH0 = LS_W1 + LS_KP1 * LS_H * 8;     // [34 kp][LS_RP rows][2]: kp 0,1 = x_t ; 2..33 = h0
constexpr int LS_H1 = LS_XH0 + LS_KP0 * LS_RP * 2;    // [32 kp][LS_RP rows][2]
constexpr int LS_HW = LS_H1 + 32 * LS_RP * 2;           // hid2act weights [2][64]
constexpr int LS_END = LS_HW + 2 * LS_H;
constexpr size_t LS_SMEM = (size_t)LS_END * sizeof(float);

__device__ __forceinline__ uint64_t pk2(float a, float b) { uint64_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ void upk2(uint64_t p, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(p)); }
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) { uint64_t r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }

__device__ __forceinline__ float rcp_apx(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float sigmoid_fast(float x) { return rcp_apx(1.0f + __expf(-x)); }
__device__ __forceinline__ float tanh_acc(float x) {
  // |x| < 0.1: odd Taylor polynomial (error < 3e-11); otherwise 1 - 2 / (1 + e^{2x}) (no cancellation there)
  const float x2 = x * x;
  const float p = x * fmaf(x2, fmaf(x2, fmaf(x2, -17.0f / 315.0f, 2.0f / 15.0f), -1.0f / 3.0f), 1.0f);
  const float e = __expf(2.0f * x);
  const float r = 1.0f - 2.0f * rcp_apx(1.0f + e);
  return fabsf(x) < 0.1f ? p : r;
}
}  // namespace


struct Lstm2Args {
  const float *z, *h0, *curr;            // [R,T,4], [R,64] (cond2hidden output), [R,4]
  const float *w0p, *w1p, *b0, *b1;      // packed weights, summed biases [256]
  const float *h2a_w, *h2a_b;
  float *act_out, *traj_out, *stash;
  int R, T;
  DynParams2 dyn;
};

// packs [in][4H] (transposed nn.LSTM weights) into [k pair][gate half][unit][2 gates][2 k]
__global__ void lstm_pack_kernel(const float* __restrict__ wihT, int in_dim, const float* __restrict__ whhT, float* __restrict__ out, int K) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= K * 256) return;
  // layout [k pair][gate half][unit][(gate lo k0, gate lo k1, gate hi k0, gate hi k1)]: conflict-free LDS.128 per warp
  int j = idx & 1, gl = (idx >> 1) & 1, u = (idx >> 2) & 63, gh = (idx >> 8) & 1, kp = idx >> 9;
  int g = gh * 2 + gl;
  int k = 2 * kp + j;
  out[idx] = (k < in_dim) ? wihT[(size_t)k * 256 + g * 64 + u] : whhT[(size_t)(k - in_dim) * 256 + g * 64 + u];
}

// h0[r][u] = cond2hidden(cond[r]) (models/vae/lstm_vae.py:46-47): step-invariant, computed once per cond tensor
__global__ void __launch_bounds__(256) lstm_h0_kernel(const float* __restrict__ cond, const float* __restrict__ c2hT,
                                                      const float* __restrict__ c2h_b, float* __restrict__ h0, int R, int C) {
  __shared__ float cs[4][256];
  const int r0 = blockIdx.x * 4, tid = threadIdx.x;
  for (int i = tid; i < 4 * C; i += 256) {
    int b = i / C, k = i - b * C;
    cs[b][k] = (r0 + b < R) ? cond[(size_t)(r0 + b) * C + k] : 0.f;
  }
  __syncthreads();
  const int b = tid >> 6, u = tid & 63;
  float acc = c2h_b[u];
  for (int k = 0; k < C; ++k) acc = fmaf(c2hT[k * LS_H + u], cs[b][k], acc);
  if (r0 + b < R) h0[(size_t)(r0 + b) * LS_H + u] = acc;
}


// acc[r][g] += sum over `nkp` k pairs of h[row r][k] * W[k][gate g] for the thread's unit
__device__ __forceinline__ void lstm_kloop(const float* __restrict__ wp, const float* __restrict__ hsrc, int nkp, uint64_t (&acc)[8][4]) {
#pragma unroll 2
  for (int kp = 0; kp < nkp; ++kp) {
    // 64-bit register pairs straight from LDS.128: (k0, k1) of one gate / one row -- no repacking moves
    const ulonglong2 wa = *reinterpret_cast<const ulonglong2*>(wp + kp * (LS_H * 8));               // (i, f)
    const ulonglong2 wb = *reinterpret_cast<const ulonglong2*>(wp + kp * (LS_H * 8) + LS_H * 4);    // (g, o)
    const ulonglong2* hp = reinterpret_cast<const ulonglong2*>(hsrc + (size_t)kp * (LS_RP * 2));
#pragma unroll
    for (int r2 = 0; r2 < 4; ++r2) {
      const ulonglong2 hv = hp[r2];                // two rows
      acc[2 * r2][0] = fma2(hv.x, wa.x, acc[2 * r2][0]); acc[2 * r2][1] = fma2(hv.x, wa.y, acc[2 * r2][1]);
      acc[2 * r2][2] = fma2(hv.x, wb.x, acc[2 * r2][2]); acc[2 * r2][3] = fma2(hv.x, wb.y, acc[2 * r2][3]);
      acc[2 * r2 + 1][0] = fma2(hv.y, wa.x, acc[2 * r2 + 1][0]); acc[2 * r2 + 1][1] = fma2(hv.y, wa.y, acc[2 * r2 + 1][1]);
      acc[2 * r2 + 1][2] = fma2(hv.y, wb.x, acc[2 * r2 + 1][2]); acc[2 * r2 + 1][3] = fma2(hv.y, wb.y, acc[2 * r2 + 1][3]);
    }
  }
}

// LSTM cell update of one layer for the thread's 8 rows; returns the new hidden values, optionally stashes
// (st = &stash[stash_index(layer, t, T, R, first row, 0, u)]: value v of the 8 rows is 8 consecutive floats at v * STASH_V_STRIDE)
template <bool SAVE>
__device__ __forceinline__ void lstm_cell(const uint64_t (&acc)[8][4], const float (&b)[4], float (&c)[8], float (&hn)[8],
                                          float* __restrict__ st) {
  float sv[5][8];
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    float x0, x1;
    upk2(acc[r][0], x0, x1); const float ig = sigmoid_fast(x0 + x1 + b[0]);
    upk2(acc[r][1], x0, x1); const float fg = sigmoid_fast(x0 + x1 + b[1]);
    upk2(acc[r][2], x0, x1); const float gg = tanh_acc(x0 + x1 + b[2]);
    upk2(acc[r][3], x0, x1); const float og = sigmoid_fast(x0 + x1 + b[3]);
    const float cn = fmaf(fg, c[r], ig * gg);
    c[r] = cn;
    hn[r] = og * tanh_acc(cn);
    if (SAVE) { sv[0][r] = ig; sv[1][r] = fg; sv[2][r] = gg; sv[3][r] = og; sv[4][r] = cn; }
  }
  if (SAVE) {
#pragma unroll
    for (int v = 0; v < 5; ++v) {
      float4* d = reinterpret_cast<float4*>(st + (size_t)v * STASH_V_STRIDE);
      d[0] = make_float4(sv[v][0], sv[v][1], sv[v][2], sv[v][3]);
      d[1] = make_float4(sv[v][4], sv[v][5], sv[v][6], sv[v][7]);
    }
  }
}

template <bool SAVE>
__global__ void __launch_bounds__(LS_THREADS, 1) lstm_decode2_kernel(const Lstm2Args a) {
  extern __shared__ __align__(16) float sm[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int rg = warp >> 1, u = (warp & 1) * 32 + lane;
  const int row0 = blockIdx.x * LS_RB, rl0 = rg * 8;     // CTA's first global row, thread's first local row
  const int T = a.T, R = a.R;
  float* xh0 = sm + LS_XH0;
  float* h1s = sm + LS_H1;

  // ---- weights -> shared memory; initial state
  {
    const float4* s0 = reinterpret_cast<const float4*>(a.w0p);
    const float4* s1 = reinterpret_cast<const float4*>(a.w1p);
    float4* d0 = reinterpret_cast<float4*>(sm + LS_W0);
    float4* d1 = reinterpret_cast<float4*>(sm + LS_W1);
    for (int i = tid; i < LS_KP0 * LS_H * 2; i += LS_THREADS) d0[i] = s0[i];
    for (int i = tid; i < LS_KP1 * LS_H * 2; i += LS_THREADS) d1[i] = s1[i];
    for (int i = tid; i < LS_RB * LS_H; i += LS_THREADS) {
      const int rl = i >> 6, k = i & 63;
      const float v = (row0 + rl < R) ? a.h0[(size_t)(row0 + rl) * LS_H + k] : 0.f;
      xh0[((2 + (k >> 1)) * LS_RP + rl) * 2 + (k & 1)] = v;
      h1s[((k >> 1) * LS_RP + rl) * 2 + (k & 1)] = v;
    }
    if (tid < 2 * LS_H) sm[LS_HW + tid] = a.h2a_w[tid];
    if (tid < LS_RB) {
      float4 zv = make_float4(0.f, 0.f, 0.f, 0.f);
      if (row0 + tid < R) zv = reinterpret_cast<const float4*>(a.z)[(size_t)(row0 + tid) * T];
      xh0[(0 * LS_RP + tid) * 2 + 0] = zv.x; xh0[(0 * LS_RP + tid) * 2 + 1] = zv.y;
      xh0[(1 * LS_RP + tid) * 2 + 0] = zv.z; xh0[(1 * LS_RP + tid) * 2 + 1] = zv.w;
    }
  }
  const float bias0[4] = {a.b0[u], a.b0[64 + u], a.b0[128 + u], a.b0[192 + u]};
  const float bias1[4] = {a.b1[u], a.b1[64 + u], a.b1[128 + u], a.b1[192 + u]};
  float c0[8], c1[8];
#pragma unroll
  for (int r = 0; r < 8; ++r) { c0[r] = 0.f; c1[r] = 0.f; }
  const float h2a_b_o = a.h2a_b[(tid >> 1) & 1];
  const float* wp0 = sm + LS_W0 + u * 4;
  const float* wp1 = sm + LS_W1 + u * 4;
  __syncthreads();

  for (int it = 0; it <= T; ++it) {
    // prefetch x_{it+1} (one row per thread of warp 0)
    float4 zn = make_float4(0.f, 0.f, 0.f, 0.f);
    if (tid < LS_RB && it + 1 < T && row0 + tid < R) zn = reinterpret_cast<const float4*>(a.z)[(size_t)(row0 + tid) * T + it + 1];
    float hn0[8], hn1[8];
    if (it < T) {                                         // layer 0, step it: [x_it | h0_{it-1}]
      uint64_t acc[8][4];
#pragma unroll
      for (int r = 0; r < 8; ++r)
#pragma unroll
        for (int g = 0; g < 4; ++g) acc[r][g] = 0ull;
      lstm_kloop(wp0, xh0 + rl0 * 2, LS_KP0, acc);
      lstm_cell<SAVE>(acc, bias0, c0, hn0, SAVE ? a.stash + stash_index(0, it, T, R, row0 + rl0, 0, u) : nullptr);
    }
    if (it >= 1) {                                        // layer 1, step it - 1: [h0_{it-1} | h1_{it-2}]
      uint64_t acc[8][4];
#pragma unroll
      for (int r = 0; r < 8; ++r)
#pragma unroll
        for (int g = 0; g < 4; ++g) acc[r][g] = 0ull;
      lstm_kloop(wp1, xh0 + (size_t)2 * (LS_RP * 2) + rl0 * 2, 32, acc);
      lstm_kloop(wp1 + 32 * (LS_H * 8), h1s + rl0 * 2, 32, acc);
      lstm_cell<SAVE>(acc, bias1, c1, hn1, SAVE ? a.stash + stash_index(1, it - 1, T, R, row0 + rl0, 0, u) : nullptr);
    }
    __syncthreads();     // every read of the state tiles of this iteration is done
    if (it < T) {
      float* hdst = xh0 + (size_t)(2 + (u >> 1)) * (LS_RP * 2) + (u & 1) + rl0 * 2;
#pragma unroll
      for (int r = 0; r < 8; ++r) hdst[r * 2] = hn0[r];
    }
    if (it >= 1) {
      float* hdst = h1s + (size_t)(u >> 1) * (LS_RP * 2) + (u & 1) + rl0 * 2;
#pragma unroll
      for (int r = 0; r < 8; ++r) hdst[r * 2] = hn1[r];
    }
    if (tid < LS_RB && it + 1 < T) {
      xh0[(0 * LS_RP + tid) * 2 + 0] = zn.x; xh0[(0 * LS_RP + tid) * 2 + 1] = zn.y;
      xh0[(1 * LS_RP + tid) * 2 + 0] = zn.z; xh0[(1 * LS_RP + tid) * 2 + 1] = zn.w;
    }
    __syncthreads();     // new states visible
    // hid2act for step it - 1 (layer 1's fresh state): the 128 layer-0 threads, (row, output, k half) each
    if (it >= 1 && tid < 128) {
      const int kh = tid & 1, o = (tid >> 1) & 1, rl = tid >> 2;
      const float* hw = sm + LS_HW + o * LS_H + kh * 32;
      const float* hs = h1s + ((size_t)(kh * 16) * LS_RP + rl) * 2;
      float s0 = 0.f, s1 = 0.f;
#pragma unroll
      for (int kp = 0; kp < 16; ++kp) {
        const float2 hv = *reinterpret_cast<const float2*>(hs + (size_t)kp * (LS_RP * 2));
        const float2 wv = *reinterpret_cast<const float2*>(hw + 2 * kp);
        s0 = fmaf(wv.x, hv.x, s0); s1 = fmaf(wv.y, hv.y, s1);
      }
      float sacc = s0 + s1;
      sacc += __shfl_xor_sync(0xffffffffu, sacc, 1);
      if (kh == 0 && row0 + rl < R) a.act_out[((size_t)(row0 + rl) * T + (it - 1)) * 2 + o] = sacc + h2a_b_o;
    }
  }
  __syncthreads();
  // ---- de-scale + unicycle closed form, one row per thread (diffuser_helpers.py:573-639)
  if (tid < LS_RB && row0 + tid < R && a.traj_out) {
    const DynParams2& d = a.dyn;
    const size_t row = (size_t)row0 + tid;
    const float* act = a.act_out + row * T * 2;
    float x = a.curr[row * 4 + 0], y = a.curr[row * 4 + 1], s = a.curr[row * 4 + 2], psi = a.curr[row * 4 + 3];
    float vprev = clip2(s, d.v_lo, d.v_hi);
    float* out = a.traj_out + row * T * 6;
    for (int k = 0; k < T; ++k) {
      const float2 av = *reinterpret_cast<const float2*>(act + k * 2);
      const float a_raw = __fadd_rn(__fmul_rn(av.x, d.a_std), d.a_mean);
      const float w_raw = __fadd_rn(__fmul_rn(av.y, d.w_std), d.w_mean);
      const float ac = clip2(a_raw, d.acce_lo, d.acce_hi);
      s = __fadd_rn(s, __fmul_rn(ac, d.dt));
      const float vnext = clip2(s, d.v_lo, d.v_hi);
      const float vbar = __fmul_rn(0.5f, __fadd_rn(vprev, vnext));
      const float ve = fabsf(vprev);
      const float yb = fmaxf(fminf(__fmul_rn(d.max_steer, ve), __fdiv_rn(d.max_yawvel, fmaxf(ve, 0.1f))), 0.1f);
      const float w = clip2(w_raw, -yb, yb);
      x = __fadd_rn(x, __fmul_rn(__fmul_rn(vbar, cosf(psi)), d.dt));
      y = __fadd_rn(y, __fmul_rn(__fmul_rn(vbar, sinf(psi)), d.dt));
      psi = __fadd_rn(psi, __fmul_rn(w, d.dt));
      float* o = out + (size_t)k * 6;
      o[0] = x; o[1] = y; o[2] = vnext; o[3] = psi; o[4] = a_raw; o[5] = w_raw;
      vprev = vnext;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// backward: d(traj) -> d(scaled actions) -> BPTT through both layers -> dz -> optimizer step
// (PerturbationGuidance.perturb, reference src/tbsim/utils/guidance_loss.py:2250-2278).  Same tiling as the
// forward: one CTA owns 32 rows; pass 1 walks layer 1 backwards in time with [W_hh1 | W_ih1]^T in shared memory
// (per step: gate gradients [32 x 256] x [256 x 128] -> recurrent dh1 (kept in registers by the thread that needs it
// next) and dh0 (to a global workspace)), pass 2 does the same for layer 0 with [W_hh0 | W_ih0]^T and emits dz.
// ------------------------------------------------------------------------------------------------
namespace {
constexpr int LB_W = 0;                                   // [128 jp][128 col][2] (pass 2: [128 jp][68 col][2])
constexpr int LB_DG = LB_W + 128 * 128 * 2;               // [128 jp][LS_RP rows][2] gate gradients
constexpr int LB_HW = LB_DG + 128 * LS_RP * 2;            // hid2act weights [2][64]
constexpr int LB_DACT = LB_HW + 2 * LS_H;                 // [32 rows][T][4]: d(action) in pass 1, dz in pass 2
static size_t lb_smem(int T) { return (size_t)(LB_DACT + LS_RB * T * 4) * sizeof(float); }
static_assert(128 * 128 * 2 >= LS_RB * 4 * (CLD_MAX_T + 1), "unicycle scratch aliases the weight tile");
}  // namespace

struct Bwd2Args {
  const float *z_mean, *act, *curr, *dtraj, *stash, *dacc;
  const float *w1t, *w0t, *h2a_w;
  float *z_out, *grad_out, *dh0f;
  int R, T;
  DynParams2 dyn;
  int optimizer; float lr;
  GuideOpt opt;                         // iteration and Adam moments of a multi-step guided call
};

// packs W_hh [256][64] | W_ih [256][in] (nn.LSTM layouts) into [j pair][col][2], col < 64: W_hh[j][col], else W_ih[j][col-64]
__global__ void lstm_pack_t_kernel(const float* __restrict__ whh, const float* __restrict__ wih, int in_dim, float* __restrict__ out) {
  const int ncol = 64 + in_dim;
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 128 * ncol * 2) return;
  int jj = idx & 1, col = (idx >> 1) % ncol, jp = (idx >> 1) / ncol;
  int j = 2 * jp + jj;
  out[idx] = (col < 64) ? whh[(size_t)j * 64 + col] : wih[(size_t)j * in_dim + (col - 64)];
}


// 8 consecutive rows of stash value v (i, f, g, o, c) of (layer, t, unit u): two 16-byte loads
__device__ __forceinline__ void stash_ld8(const float* __restrict__ stash, int layer, int t, int T, int R, int row, int v, int u, float (&o)[8]) {
  const float4* p = reinterpret_cast<const float4*>(stash + stash_index(layer, t, T, R, row, v, u));
  const float4 a = p[0], b = p[1];
  o[0] = a.x; o[1] = a.y; o[2] = a.z; o[3] = a.w; o[4] = b.x; o[5] = b.y; o[6] = b.z; o[7] = b.w;
}

__global__ void __launch_bounds__(LS_THREADS, 1) lstm_backward2_kernel(const Bwd2Args a) {
  extern __shared__ __align__(16) float sm[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int rg = warp >> 1, u = (warp & 1) * 32 + lane;
  const int row0 = blockIdx.x * LS_RB, rl0 = rg * 8;
  const int T = a.T, R = a.R;
  float* dg = sm + LB_DG;
  float* dact = sm + LB_DACT;      // pass 1: d(scaled action) [32][T][2]
  float* dzs = sm + LB_DACT;       // pass 2: dz [32][T][4] (same storage)

  // ---- unicycle backward per row -> dact (scratch aliases the weight tile); then layer-1 weights -> smem
  {
    if (tid < 2 * LS_H) sm[LB_HW + tid] = a.h2a_w[tid];
    if (tid < LS_RB) {
      float* da = dact + tid * T * 2;
      if (row0 + tid < R) {
        const size_t row = (size_t)row0 + tid;
        unicycle_row_backward2(a.act + row * T * 2, a.curr + row * 4, a.dtraj + row * T * 4, T, a.dyn, sm + LB_W + tid * 4 * (T + 1), da,
                               a.dacc ? a.dacc + row * T : nullptr);
      } else {
        for (int i = 0; i < 2 * T; ++i) da[i] = 0.f;
      }
    }
    __syncthreads();
    const float4* s1 = reinterpret_cast<const float4*>(a.w1t);
    float4* d1 = reinterpret_cast<float4*>(sm + LB_W);
    for (int i = tid; i < 128 * 128 * 2 / 4; i += LS_THREADS) d1[i] = s1[i];
  }
  __syncthreads();
  const float hw0 = sm[LB_HW + u], hw1 = sm[LB_HW + LS_H + u];
  const bool rv[8] = {row0 + rl0 + 0 < R, row0 + rl0 + 1 < R, row0 + rl0 + 2 < R, row0 + rl0 + 3 < R,
                      row0 + rl0 + 4 < R, row0 + rl0 + 5 < R, row0 + rl0 + 6 < R, row0 + rl0 + 7 < R};

  // =========================== pass 1: layer 1 ===========================
  {
    const int frow = row0 + rl0;                                                // rows beyond R read the zero-padded / stale tail: masked by rv
    float gi[8], gf[8], gg[8], go[8], cc[8], cp[8];                              // gates of step t, c(t), c(t-1)
    float dhrec[8], dcrec[8];
    stash_ld8(a.stash, 1, T - 1, T, R, frow, 0, u, gi); stash_ld8(a.stash, 1, T - 1, T, R, frow, 1, u, gf);
    stash_ld8(a.stash, 1, T - 1, T, R, frow, 2, u, gg); stash_ld8(a.stash, 1, T - 1, T, R, frow, 3, u, go);
    stash_ld8(a.stash, 1, T - 1, T, R, frow, 4, u, cc);
    if (T >= 2) stash_ld8(a.stash, 1, T - 2, T, R, frow, 4, u, cp);
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      dhrec[r] = 0.f; dcrec[r] = 0.f;
      if (T < 2) cp[r] = 0.f;
    }
    for (int t = T - 1; t >= 0; --t) {
      // prefetch: gates of t-1, cell of t-2
      float ni[8], nf[8], ng[8], no[8], np[8];
      if (t >= 1) {
        stash_ld8(a.stash, 1, t - 1, T, R, frow, 0, u, ni); stash_ld8(a.stash, 1, t - 1, T, R, frow, 1, u, nf);
        stash_ld8(a.stash, 1, t - 1, T, R, frow, 2, u, ng); stash_ld8(a.stash, 1, t - 1, T, R, frow, 3, u, no);
      }
      if (t >= 2) stash_ld8(a.stash, 1, t - 2, T, R, frow, 4, u, np);
      else {
#pragma unroll
        for (int r = 0; r < 8; ++r) np[r] = 0.f;
      }
      // gate gradients of step t
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const float2 da = *reinterpret_cast<const float2*>(dact + ((rl0 + r) * T + t) * 2);
        const float dh = fmaf(hw0, da.x, fmaf(hw1, da.y, dhrec[r]));
        const float tc = tanh_acc(cc[r]);
        const float dc = dcrec[r] + dh * go[r] * (1.f - tc * tc);
        float* d = dg + (size_t)(rl0 + r) * 2 + (u & 1) + (size_t)(u >> 1) * (LS_RP * 2);
        d[0 * 32 * (LS_RP * 2)] = dc * gg[r] * gi[r] * (1.f - gi[r]);
        d[1 * 32 * (LS_RP * 2)] = dc * cp[r] * gf[r] * (1.f - gf[r]);
        d[2 * 32 * (LS_RP * 2)] = dc * gi[r] * (1.f - gg[r] * gg[r]);
        d[3 * 32 * (LS_RP * 2)] = dh * tc * go[r] * (1.f - go[r]);
        dcrec[r] = dc * gf[r];
      }
      __syncthreads();
      // [32 x 256] x [256 x 128]: this thread: 8 rows x columns (u: W_hh1^T -> dh1 recurrent, 64+u: W_ih1^T -> dh0)
      uint64_t acc[8][2];
#pragma unroll
      for (int r = 0; r < 8; ++r) { acc[r][0] = 0ull; acc[r][1] = 0ull; }
      {
        const float* wp = sm + LB_W + u * 2;
        const float* gp = dg + rl0 * 2;
#pragma unroll 4
        for (int jp = 0; jp < 128; ++jp) {
          const uint64_t w_a = *reinterpret_cast<const uint64_t*>(wp + jp * 256);
          const uint64_t w_b = *reinterpret_cast<const uint64_t*>(wp + jp * 256 + 128);
          const ulonglong2* hp = reinterpret_cast<const ulonglong2*>(gp + (size_t)jp * (LS_RP * 2));
#pragma unroll
          for (int r2 = 0; r2 < 4; ++r2) {
            const ulonglong2 hv = hp[r2];
            acc[2 * r2][0] = fma2(hv.x, w_a, acc[2 * r2][0]); acc[2 * r2][1] = fma2(hv.x, w_b, acc[2 * r2][1]);
            acc[2 * r2 + 1][0] = fma2(hv.y, w_a, acc[2 * r2 + 1][0]); acc[2 * r2 + 1][1] = fma2(hv.y, w_b, acc[2 * r2 + 1][1]);
          }
        }
      }
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        float x0, x1;
        upk2(acc[r][0], x0, x1); dhrec[r] = x0 + x1;
        upk2(acc[r][1], x0, x1);
        if (rv[r]) a.dh0f[((size_t)t * R + row0 + rl0 + r) * LS_H + u] = x0 + x1;
        gi[r] = ni[r]; gf[r] = nf[r]; gg[r] = ng[r]; go[r] = no[r]; cc[r] = cp[r]; cp[r] = np[r];
      }
      __syncthreads();
    }
  }
  // =========================== pass 2: layer 0 ===========================
  {
    const float4* s0 = reinterpret_cast<const float4*>(a.w0t);
    float4* d0 = reinterpret_cast<float4*>(sm + LB_W);
    for (int i = tid; i < 128 * 68 * 2 / 4; i += LS_THREADS) d0[i] = s0[i];
    __threadfence_block();
    __syncthreads();
    const int frow = row0 + rl0;
    float gi[8], gf[8], gg[8], go[8], cc[8], cp[8], dhf[8];
    float dhrec[8], dcrec[8];
    stash_ld8(a.stash, 0, T - 1, T, R, frow, 0, u, gi); stash_ld8(a.stash, 0, T - 1, T, R, frow, 1, u, gf);
    stash_ld8(a.stash, 0, T - 1, T, R, frow, 2, u, gg); stash_ld8(a.stash, 0, T - 1, T, R, frow, 3, u, go);
    stash_ld8(a.stash, 0, T - 1, T, R, frow, 4, u, cc);
    if (T >= 2) stash_ld8(a.stash, 0, T - 2, T, R, frow, 4, u, cp);
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      dhrec[r] = 0.f; dcrec[r] = 0.f;
      if (T < 2) cp[r] = 0.f;
      dhf[r] = rv[r] ? a.dh0f[((size_t)(T - 1) * R + row0 + rl0 + r) * LS_H + u] : 0.f;
    }
    for (int t = T - 1; t >= 0; --t) {
      float ni[8], nf[8], ng[8], no[8], np[8], nh[8];
      if (t >= 1) {
        stash_ld8(a.stash, 0, t - 1, T, R, frow, 0, u, ni); stash_ld8(a.stash, 0, t - 1, T, R, frow, 1, u, nf);
        stash_ld8(a.stash, 0, t - 1, T, R, frow, 2, u, ng); stash_ld8(a.stash, 0, t - 1, T, R, frow, 3, u, no);
      }
      if (t >= 2) stash_ld8(a.stash, 0, t - 2, T, R, frow, 4, u, np);
      else {
#pragma unroll
        for (int r = 0; r < 8; ++r) np[r] = 0.f;
      }
#pragma unroll
      for (int r = 0; r < 8; ++r) nh[r] = (rv[r] && t >= 1) ? a.dh0f[((size_t)(t - 1) * R + row0 + rl0 + r) * LS_H + u] : 0.f;
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const float dh = dhf[r] + dhrec[r];
        const float tc = tanh_acc(cc[r]);
        const float dc = dcrec[r] + dh * go[r] * (1.f - tc * tc);
        float* d = dg + (size_t)(rl0 + r) * 2 + (u & 1) + (size_t)(u >> 1) * (LS_RP * 2);
        d[0 * 32 * (LS_RP * 2)] = dc * gg[r] * gi[r] * (1.f - gi[r]);
        d[1 * 32 * (LS_RP * 2)] = dc * cp[r] * gf[r] * (1.f - gf[r]);
        d[2 * 32 * (LS_RP * 2)] = dc * gi[r] * (1.f - gg[r] * gg[r]);
        d[3 * 32 * (LS_RP * 2)] = dh * tc * go[r] * (1.f - go[r]);
        dcrec[r] = dc * gf[r];
      }
      __syncthreads();
      // [32 x 256] x [256 x 68]: column u (W_hh0^T -> dh0 recurrent); threads with u < 4 also column 64+u (W_ih0^T -> dz)
      uint64_t acc[8], accz[8];
#pragma unroll
      for (int r = 0; r < 8; ++r) { acc[r] = 0ull; accz[r] = 0ull; }
      {
        const float* wp = sm + LB_W + u * 2;
        const float* gp = dg + rl0 * 2;
        const bool zc = u < 4;                              // warp-uniform only for the second warp of a row group (never)
#pragma unroll 4
        for (int jp = 0; jp < 128; ++jp) {
          const uint64_t w_a = *reinterpret_cast<const uint64_t*>(wp + jp * 136);
          uint64_t w_z = 0ull;
          if (zc) w_z = *reinterpret_cast<const uint64_t*>(wp + jp * 136 + 128);
          const ulonglong2* hp = reinterpret_cast<const ulonglong2*>(gp + (size_t)jp * (LS_RP * 2));
#pragma unroll
          for (int r2 = 0; r2 < 4; ++r2) {
            const ulonglong2 hv = hp[r2];
            acc[2 * r2] = fma2(hv.x, w_a, acc[2 * r2]); acc[2 * r2 + 1] = fma2(hv.y, w_a, acc[2 * r2 + 1]);
            if (zc) { accz[2 * r2] = fma2(hv.x, w_z, accz[2 * r2]); accz[2 * r2 + 1] = fma2(hv.y, w_z, accz[2 * r2 + 1]); }
          }
        }
      }
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        float x0, x1;
        upk2(acc[r], x0, x1); dhrec[r] = x0 + x1;
        if (u < 4) {
          upk2(accz[r], x0, x1);
          dzs[((rl0 + r) * T + t) * 4 + u] = x0 + x1;       // staged; the optimizer step runs after the loop
        }
        gi[r] = ni[r]; gf[r] = nf[r]; gg[r] = ng[r]; go[r] = no[r]; cc[r] = cp[r]; cp[r] = np[r]; dhf[r] = nh[r];
      }
      __syncthreads();
    }
    // ---- optimizer step (guidance_loss.py:2250-2278), coalesced over the CTA's [32][T][4] block
    for (int i = tid; i < LS_RB * T * 4; i += LS_THREADS) {
      const int rl = i / (T * 4);
      if (row0 + rl >= R) continue;
      const size_t gi_ = (size_t)row0 * T * 4 + i;
      const float g = dzs[i], z = a.z_mean[gi_];
      float zn;
      if (a.optimizer == CLD_OPT_ADAM) {
        float m, v;
        if (!a.opt.m) {
          zn = adam_first_step(z, g, a.lr, m, v);
        } else {
          // multi-step call: the moments live across iterations
          if (a.opt.iter == 1) {
            zn = adam_first_step(z, g, a.lr, m, v);
          } else {
            m = a.opt.m[gi_]; v = a.opt.v[gi_];
            zn = adam_next_step(z, g, a.opt.step_size, a.opt.bc2_sqrt, m, v);
          }
          a.opt.m[gi_] = m; a.opt.v[gi_] = v;
        }
      } else {
        zn = z - a.lr * g;
      }
      a.z_out[gi_] = zn;
      if (a.grad_out) a.grad_out[gi_] = g;
    }
  }
}

// prepares the packed weights on first use
static int lstm2_prepare(CldHandle* h, cudaStream_t s) {
  DecoderW& w = h->dec;
  if (w.w0p) return 0;
  float *w0p = nullptr, *w1p = nullptr;
  CLD_CUDA_OK(h, cudaMalloc((void**)&w0p, (size_t)LS_KP0 * LS_H * 8 * sizeof(float)));
  h->allocs.push_back(w0p);
  CLD_CUDA_OK(h, cudaMalloc((void**)&w1p, (size_t)LS_KP1 * LS_H * 8 * sizeof(float)));
  h->allocs.push_back(w1p);
  lstm_pack_kernel<<<(2 * LS_KP0 * 256 + 255) / 256, 256, 0, s>>>(w.wih0, 4, w.whh0, w0p, 2 * LS_KP0);
  lstm_pack_kernel<<<(2 * LS_KP1 * 256 + 255) / 256, 256, 0, s>>>(w.wih1, 64, w.whh1, w1p, 2 * LS_KP1);
  CLD_LAUNCH_OK(h, "lstm_pack_kernel");
  CLD_CUDA_OK(h, cudaFuncSetAttribute(lstm_decode2_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LS_SMEM));
  CLD_CUDA_OK(h, cudaFuncSetAttribute(lstm_decode2_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LS_SMEM));
  float *w1t = nullptr, *w0t = nullptr;
  CLD_CUDA_OK(h, cudaMalloc((void**)&w1t, (size_t)128 * 128 * 2 * sizeof(float)));
  h->allocs.push_back(w1t);
  CLD_CUDA_OK(h, cudaMalloc((void**)&w0t, (size_t)128 * 68 * 2 * sizeof(float)));
  h->allocs.push_back(w0t);
  lstm_pack_t_kernel<<<(128 * 128 * 2 + 255) / 256, 256, 0, s>>>(w.whh1_raw, w.wih1_raw, 64, w1t);
  lstm_pack_t_kernel<<<(128 * 68 * 2 + 255) / 256, 256, 0, s>>>(w.whh0_raw, w.wih0_raw, 4, w0t);
  CLD_LAUNCH_OK(h, "lstm_pack_t_kernel");
  if (lb_smem(h->cfg.horizon) > 232448) return fail(h, CLD_ERR_UNSUPPORTED, "horizon too long for the LSTM backward kernel");
  CLD_CUDA_OK(h, cudaFuncSetAttribute(lstm_backward2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lb_smem(h->cfg.horizon)));
  w.w0p = w0p; w.w1p = w1p; w.w1t = w1t; w.w0t = w0t;
  return 0;
}

int decode_h0(CldHandle* h, const float* cond, float* h0, int R, cudaStream_t s) {
  const DecoderW& w = h->dec;
  if (!w.loaded) return fail(h, CLD_ERR_STATE, "decoder weights not loaded");
  lstm_h0_kernel<<<(R + 3) / 4, 256, 0, s>>>(cond, w.c2h_w, w.c2h_b, h0, R, h->cfg.cond_dim);
  CLD_LAUNCH_OK(h, "lstm_h0_kernel");
  return 0;
}

// act_out must be a valid [R,T,2] buffer (the rollout reads it back)
int decode_rollout_h0(CldHandle* h, const float* z, const float* h0, const float* curr, float* act_out, float* traj_out,
                      bool save, int R, cudaStream_t s) {
  DecoderW& w = h->dec;
  if (!w.loaded) return fail(h, CLD_ERR_STATE, "decoder weights not loaded");
  if (h->use_lstm_tc) return decode_rollout_h0_tc(h, z, h0, curr, act_out, traj_out, save, R, s);
  if (h->cfg.hidden != LS_H || h->cfg.latent_dim != 4) return fail(h, CLD_ERR_UNSUPPORTED, "decoder kernel is specialised for hidden=64, latent=4");
  int rc;
  if ((rc = lstm2_prepare(h, s))) return rc;
  const CldConfig& c = h->cfg;
  Lstm2Args a;
  a.z = z; a.h0 = h0; a.curr = curr; a.w0p = w.w0p; a.w1p = w.w1p; a.b0 = w.b0; a.b1 = w.b1;
  a.h2a_w = w.h2a_w; a.h2a_b = w.h2a_b; a.act_out = act_out; a.traj_out = traj_out; a.stash = save ? h->stash : nullptr;
  a.R = R; a.T = c.horizon;
  a.dyn.dt = c.dt; a.dyn.acce_lo = c.acce_lo; a.dyn.acce_hi = c.acce_hi; a.dyn.v_lo = c.v_lo; a.dyn.v_hi = c.v_hi;
  a.dyn.max_steer = c.max_steer; a.dyn.max_yawvel = c.max_yawvel;
  a.dyn.a_mean = c.norm_mean[4]; a.dyn.a_std = c.norm_std[4]; a.dyn.w_mean = c.norm_mean[5]; a.dyn.w_std = c.norm_std[5];
  const int grid = (R + LS_RB - 1) / LS_RB;
  if (save) lstm_decode2_kernel<true><<<grid, LS_THREADS, LS_SMEM, s>>>(a);
  else lstm_decode2_kernel<false><<<grid, LS_THREADS, LS_SMEM, s>>>(a);
  CLD_LAUNCH_OK(h, "lstm_decode2_kernel");
  return 0;
}


int decode_backward_update2(CldHandle* h, const float* z_mean, const float* act, const float* curr, const float* dtraj,
                            const float* dtraj2, const float* dacc, const CldGuidanceConfig* g, const GuideOpt& opt, float* z_out,
                            float* grad_out, int R, cudaStream_t s) {
  DecoderW& w = h->dec;
  int rc;
  if (h->use_lstm_tc && !h->env_lstm_bwd_simt)
    return decode_backward_update_tc(h, z_mean, act, curr, dtraj, dtraj2, dacc, g, opt, z_out, grad_out, R, s);
  if (dtraj2) return fail(h, CLD_ERR_STATE, "internal: split d(traj) buffers are only handled by the tensor-core backward");
  if ((rc = lstm2_prepare(h, s))) return rc;
  const CldConfig& c = h->cfg;
  if (c.horizon > CLD_MAX_T) return fail(h, CLD_ERR_UNSUPPORTED, "horizon exceeds CLD_MAX_T");
  Bwd2Args a;
  a.z_mean = z_mean; a.act = act; a.curr = curr; a.dtraj = dtraj; a.stash = h->stash; a.dacc = dacc;
  a.w1t = w.w1t; a.w0t = w.w0t; a.h2a_w = w.h2a_w; a.z_out = z_out; a.grad_out = grad_out; a.dh0f = h->ws_dh0;
  a.R = R; a.T = c.horizon;
  a.dyn.dt = c.dt; a.dyn.acce_lo = c.acce_lo; a.dyn.acce_hi = c.acce_hi; a.dyn.v_lo = c.v_lo; a.dyn.v_hi = c.v_hi;
  a.dyn.max_steer = c.max_steer; a.dyn.max_yawvel = c.max_yawvel;
  a.dyn.a_mean = c.norm_mean[4]; a.dyn.a_std = c.norm_std[4]; a.dyn.w_mean = c.norm_mean[5]; a.dyn.w_std = c.norm_std[5];
  a.optimizer = g->optimizer; a.lr = g->lr; a.opt = opt;
  lstm_backward2_kernel<<<(R + LS_RB - 1) / LS_RB, LS_THREADS, lb_smem(a.T), s>>>(a);
  CLD_LAUNCH_OK(h, "lstm_backward2_kernel");
  return 0;
}

}  // namespace cld
