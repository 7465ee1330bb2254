// Pieces shared by the SIMT (kernels_lstm.cu) and tensor-core (kernels_lstm_tc.cu) LSTM decoder kernels.
#pragma once
#include "common.cuh"

namespace cld {

struct DynParams2 {
  float dt, acce_lo, acce_hi, v_lo, v_hi, max_steer, max_yawvel;
  float a_mean, a_std, w_mean, w_std;
};

__device__ __forceinline__ float clip2(float x, float lo, float hi) { return fminf(fmaxf(x, lo), hi); }

inline DynParams2 make_dyn2(const CldConfig& c) {
  DynParams2 d;
  d.dt = c.dt; d.acce_lo = c.acce_lo; d.acce_hi = c.acce_hi; d.v_lo = c.v_lo; d.v_hi = c.v_hi;
  d.max_steer = c.max_steer; d.max_yawvel = c.max_yawvel;
  d.a_mean = c.norm_mean[4]; d.a_std = c.norm_std[4]; d.w_mean = c.norm_mean[5]; d.w_std = c.norm_std[5];
  return d;
}

// de-scale + unicycle closed form for one row (diffuser_helpers.py:573-639, vae_model.py:100-129): act [T][2] -> out [T][6]
__device__ __forceinline__ void unicycle_row_forward2(const float* act, const float* curr, int T, const DynParams2& d, float* out) {
  float x = curr[0], y = curr[1], s = curr[2], psi = curr[3];
  float vprev = clip2(s, d.v_lo, d.v_hi);
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

// reverse of the unicycle closed form for one row (SURVEY.md Appendix C); writes d(scaled action) [T][2]
// dacc: optional [T] direct gradient w.r.t. the de-scaled acceleration command (acc-limit guidance: x6[..., 4] is the command itself)
__device__ inline void unicycle_row_backward2(const float* act, const float* curr, const float* dtr, int T, const DynParams2& a,
                                       float* scr /*[4][T+1]*/, float* dact, const float* dacc = nullptr) {
  float* sk = scr; float* psik = scr + (T + 1); float* vbar = scr + 2 * (T + 1); float* msk = scr + 3 * (T + 1);
  float s = curr[2], psi = curr[3];
  float vprev = clip2(s, a.v_lo, a.v_hi);
  sk[0] = s; psik[0] = psi;
  for (int k = 0; k < T; ++k) {
    float a_raw = __fadd_rn(__fmul_rn(act[k * 2 + 0], a.a_std), a.a_mean);
    float w_raw = __fadd_rn(__fmul_rn(act[k * 2 + 1], a.w_std), a.w_mean);
    float ac = clip2(a_raw, a.acce_lo, a.acce_hi);
    s = __fadd_rn(s, __fmul_rn(ac, a.dt));
    float vnext = clip2(s, a.v_lo, a.v_hi);
    vbar[k] = __fmul_rn(0.5f, __fadd_rn(vprev, vnext));
    float ve = fabsf(vprev);
    float yb = fmaxf(fminf(__fmul_rn(a.max_steer, ve), __fdiv_rn(a.max_yawvel, fmaxf(ve, 0.1f))), 0.1f);
    float w = clip2(w_raw, -yb, yb);
    psi = __fadd_rn(psi, __fmul_rn(w, a.dt));
    int m = ((a_raw >= a.acce_lo && a_raw <= a.acce_hi) ? 1 : 0) | ((w_raw >= -yb && w_raw <= yb) ? 2 : 0);
    msk[k] = __int_as_float(m);
    sk[k + 1] = s; psik[k + 1] = psi;
    vprev = vnext;
  }
  float Gx = 0.f, Gy = 0.f, Spsi = 0.f, Ss = 0.f, dvbar_next = 0.f, direct_next = 0.f;
  for (int m = T - 1; m >= 0; --m) {
    const float gx = dtr[m * 4 + 0], gy = dtr[m * 4 + 1], gv = dtr[m * 4 + 2], gpsi = dtr[m * 4 + 3];
    Gx += a.dt * gx; Gy += a.dt * gy;
    float c = cosf(psik[m]), sn = sinf(psik[m]);
    float dvbar = Gx * c + Gy * sn;
    float direct = vbar[m] * (-Gx * sn + Gy * c);
    Spsi += ((m + 1 <= T - 1) ? direct_next : 0.f) + gpsi;
    float dvhat = 0.5f * (((m + 1 <= T - 1) ? dvbar_next : 0.f) + dvbar) + gv;
    float s1 = sk[m + 1];
    if (s1 >= a.v_lo && s1 <= a.v_hi) Ss += dvhat;
    int mk = __float_as_int(msk[m]);
    float du0 = (mk & 1) ? a.dt * Ss : 0.f;
    float du1 = (mk & 2) ? a.dt * Spsi : 0.f;
    if (dacc) du0 += dacc[m];
    dact[m * 2 + 0] = a.a_std * du0;
    dact[m * 2 + 1] = a.w_std * du1;
    dvbar_next = dvbar; direct_next = direct;
  }
}

// torch.optim.Adam (betas 0.9 / 0.999, eps 1e-8) on one element of z (guidance_loss.py:2250-2278).  First step, from zero
// moments: m = 0.1 g, v = 0.001 g^2, bias corrections 0.1 / 0.001, so the update is z - lr g / (|g| + 1e-8).
__device__ __forceinline__ float adam_first_step(float z, float g, float lr, float& m, float& v) {
  m = 0.1f * g;
  v = (0.001f * g) * g;
  const float denom = sqrtf(v) / 0.03162277660168379f + 1e-8f;
  return z - (lr / 0.1f) * (m / denom);
}
// a later step (torch's single-tensor form): m.lerp_(g, 0.1), v = 0.999 v + 0.001 g^2, z -= step_size m / (sqrt(v) / bc2_sqrt + eps)
__device__ __forceinline__ float adam_next_step(float z, float g, float step_size, float bc2_sqrt, float& m, float& v) {
  m = m + 0.1f * (g - m);
  v = v * 0.999f + (0.001f * g) * g;
  const float denom = sqrtf(v) / bc2_sqrt + 1e-8f;
  return z - step_size * (m / denom);
}

}  // namespace cld
