// Guidance gradient with an ANALYTIC backward (replaces autograd through
// PerturbationGuidance.perturb, reference src/tbsim/utils/guidance_loss.py:2221-2282):
//   guidance_loss_grad      d(loss)/d(trajectory) of AgentCollisionLoss (:505-626), MapCollisionLoss (:772-870)
//                           and TargetPosLoss (:693-712), one (scene, sample) per CTA, warp-shuffle reductions
//                           over time / sample points; normalisation = "one scene per reference call"
//                           (DiffuserGuidance.compute_guidance_loss :2143-2174).
//   decode_backward_update  unicycle backward (reverse scans, clip masks) -> hid2act^T -> LSTM BPTT
//                           (two layers, stash written by the forward kernel) -> dz, fused with the first
//                           Adam / SGD step of perturb (:2250-2278).
// All arithmetic fp32 (the update is sign-sensitive: SURVEY.md section 7, hard part 3).
#include <math.h>
#include <stdio.h>

#include "common.cuh"

namespace cld {

__device__ __forceinline__ float clipg(float x, float lo, float hi) { return fminf(fmaxf(x, lo), hi); }

struct LossArgs {
  const float* traj;     // [R,T,6]
  float* dtraj;          // [R,T,4]  d/d(x, y, v, yaw)
  float* loss;           // [7,R] or nullptr: agent_collision, map_collision, target_pos, target_speed, acc_limit, speed_limit, waypoint
  float* dacc;           // [R,T] d/d(acc) of the acc-limit term (acc = de-scaled action, not a function of the rollout) or nullptr
  const float *extent, *wfa, *rfa, *speed, *target, *tspeed;
  float w_ts, w_al, acc_limit, w_sl, speed_limit;
  // waypoint terms (per agent): local target [B,2], mode [B] (0 none | 1 at-time | 2 final-distance hinge | 3 progress hinge | 4 TargetPosLoss),
  // time step [B], goal distance [B], per-agent multiplier [B] (A / number of guided agents of the scene: the reference averages over them)
  const float *wp_target, *wp_dist, *wp_w; const int *wp_mode, *wp_time; float w_wp;
  const uint8_t* dmap; int H, W, packed;   // packed: rows of (W + 7) / 8 bytes, pixel x = bit (x & 7) of byte x >> 3
  int S, A, N, T, R;
  float w_ac, w_mc, w_tp;
  int D; float buffer, decay, speed_th, min_target_time;
  int nl, nw;
  // map-collision term: screen + work list (see guidance_map_screen_kernel)
  const uint8_t* pk; int pk_pitch;          // the drivable maps with one bit per pixel (rows of pk_pitch bytes; nullptr: no screen)
  int* work;                                // [0] items listed, [1] CTAs of the list kernel that have finished, [2...] items = row * T + t
  int exhaustive;                           // debug (CLD_MAP_EXHAUSTIVE=1): nearest on-road point by the exhaustive search only
  int assign;                               // the map term OWNS dtraj (writes every item, zeros included) instead of adding to it
  float lwise[16], wwise[16];
  float wts[CLD_MAX_T];   // decay^t / sum_t decay^t  (guidance_loss.py:607-608)
};

// torch.linspace(lo, hi, n)[i] in fp32 (symmetric evaluation, as ATen does)
__device__ __forceinline__ float linspace_at(float lo, float hi, int n, int i) {
  if (n == 1) return lo;
  float step = (hi - lo) / (float)(n - 1);
  return (i < n / 2) ? lo + step * (float)i : hi - step * (float)(n - 1 - i);
}

// TargetPosLoss.forward (guidance_loss.py:693-712) for one (agent, sample) row by one warp, lanes over time: adds kk * d(loss)/d(x, y)
// to dtraj [T,4] and returns the loss (all lanes).  tr = traj row [T,6].
__device__ __forceinline__ float target_pos_term(const float* __restrict__ tr, float* __restrict__ dtraj, float tx, float ty, int t0, int T,
                                                 int lane, float kk) {
  const int Tn = T - t0;
  float dmin = 3.4e38f;
  for (int t = t0 + lane; t < T; t += 32) {
    float dx = tr[t * 6] - tx, dy = tr[t * 6 + 1] - ty;
    dmin = fminf(dmin, sqrtf(dx * dx + dy * dy));
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) dmin = fminf(dmin, __shfl_xor_sync(0xffffffffu, dmin, o));
  float Z = 0.f, E = 0.f;
  for (int t = t0 + lane; t < T; t += 32) {
    float dx = tr[t * 6] - tx, dy = tr[t * 6 + 1] - ty;
    float d2 = dx * dx + dy * dy, d = sqrtf(d2);
    float e = expf(-(d - dmin));
    Z += e; E += e * d2;
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    Z += __shfl_xor_sync(0xffffffffu, Z, o);
    E += __shfl_xor_sync(0xffffffffu, E, o);
  }
  E /= Z;
  if (kk != 0.f) {
    const float k2 = kk / (float)Tn;
    for (int t = t0 + lane; t < T; t += 32) {
      float dx = tr[t * 6] - tx, dy = tr[t * 6 + 1] - ty;
      float d2 = dx * dx + dy * dy, d = sqrtf(d2);
      float sw = expf(-(d - dmin)) / Z;
      float f = 2.f * sw + ((d > 0.f) ? sw * (E - d2) / d : 0.f);
      dtraj[t * 4] += k2 * f * dx; dtraj[t * 4 + 1] += k2 * f * dy;
    }
  }
  return E / (float)Tn;
}

__device__ __forceinline__ bool is_moving(const LossArgs& a, size_t g) { return fabsf(a.speed[g]) > a.speed_th; }

// Agent-collision constants of agent g (its global agent index): rad, cmin, cmax, moving, R00, R01, R10, R11
__device__ __forceinline__ void collision_consts(const LossArgs& a, size_t g, float* q) {
  float L = a.extent[g * 3 + 0], Wd = a.extent[g * 3 + 1];
  float rad = Wd / 2.f;
  q[0] = rad; q[1] = -(L / 2.f) + rad; q[2] = (L / 2.f) - rad;
  q[3] = is_moving(a, g) ? 1.f : 0.f;
  q[4] = a.wfa[g * 9 + 0]; q[5] = a.wfa[g * 9 + 1]; q[6] = a.wfa[g * 9 + 3]; q[7] = a.wfa[g * 9 + 4];
}

// World pose (Px, Py, cos Psi, sin Psi) of agent g, sample n at step t: transform_agents_to_world (geometry_utils.py:458-483)
__device__ __forceinline__ float4 world_pose(const LossArgs& a, size_t g, int n, int t) {
  const float* tr = a.traj + ((g * a.N + n) * a.T + t) * 6;
  float px = tr[0], py = tr[1], psi = tr[3];
  const float* M = a.wfa + g * 9;
  float Px = M[0] * px + M[1] * py + M[2], Py = M[3] * px + M[4] * py + M[5];
  float c = cosf(psi), sn = sinf(psi);
  float hx = M[0] * c + M[1] * sn, hy = M[3] * c + M[4] * sn;
  float Psi = atan2f(hy, hx);
  return make_float4(Px, Py, cosf(Psi), sinf(Psi));
}

// Stage partners [g0, g0 + nt) of sample n at steps [t0, t0 + nts): poses [nt][ts][4] (ts >= nts steps per partner) and
// constants [nt][8]
__device__ __forceinline__ void stage_partners(const LossArgs& a, float* pose, float* agt, size_t g0, int nt, int n, int t0, int nts,
                                               int ts) {
  const int tid = threadIdx.x, nthr = blockDim.x;
  for (int j = tid; j < nt; j += nthr) collision_consts(a, g0 + j, agt + j * 8);
  for (int it = tid; it < nt * nts; it += nthr) {
    const int j = it / nts, t = it - j * nts;
    reinterpret_cast<float4*>(pose)[(size_t)j * ts + t] = world_pose(a, g0 + j, n, t0 + t);
  }
}

// Agent-collision partners in shared memory: a scene of up to SCENE_TILE agents is staged whole, a larger one streams tiles of
// PARTNER_TILE agents x 32 steps
constexpr int SCENE_TILE = 64, PARTNER_TILE = 128;

__global__ void __launch_bounds__(512) guidance_loss_grad_kernel(LossArgs a) {
  extern __shared__ __align__(16) float sm[];
  const int A = a.A, T = a.T, N = a.N;
  // The partners j of the agent-collision term pass through shared memory in tiles.  A scene of at most SCENE_TILE agents is
  // one tile holding all its steps, staged once.  A larger scene is streamed as tiles of PARTNER_TILE partners x the 32 steps
  // of one lane slot, so shared memory does not depend on A.  Tiles go in ascending j: every sum over partners is added in the
  // same order whatever the tiling.
  const bool one_tile = A <= SCENE_TILE;
  const int P = one_tile ? A : PARTNER_TILE, TS = one_tile ? T : 32;
  float* pose = sm;                         // [P][TS][4] world Px, Py, cos(Psi), sin(Psi) of the tile's partners
  float* agt = pose + (size_t)P * TS * 4;   // [P][8]: rad, cmin, cmax, moving, R00, R01, R10, R11
  float* wts = agt + P * 8;                 // [T] decay weights
  const int s = blockIdx.x / N, n = blockIdx.x % N;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int nthr = blockDim.x, nwarps = nthr >> 5;       // 16 warps: one agent per warp at 16 agents per scene (latency-bound loops: more warps per SM)
  // the agents of a scene are dealt to gridDim.y CTAs (large scenes: 64 agents x 104 steps x 63 partners would otherwise sit on
  // S * N CTAs); every CTA visits the poses of ALL agents (the partners) and evaluates the terms of agents [i_lo, i_hi)
  const int per_cta = (A + (int)gridDim.y - 1) / (int)gridDim.y;
  const int i_lo = (int)blockIdx.y * per_cta, i_hi = min(A, i_lo + per_cta);
  const size_t ag0 = (size_t)s * A;
  const float inv_AN = 1.0f / (float)(A * N);

  for (int t = tid; t < T; t += nthr) wts[t] = a.wts[t];
  if (one_tile) stage_partners(a, pose, agt, ag0, A, n, 0, T, T);
  __syncthreads();

  // ---------------- agent-agent collision: warp per agent, lanes over time ---------------------
  // Loops that stage tiles are CTA-uniform: every warp runs all rounds and slots.  With several tiles the host deals at most one
  // agent to a warp (one round), so each tile is staged once per CTA.
  const int rounds = i_hi > i_lo ? (i_hi - i_lo + nwarps - 1) / nwarps : 0;
  for (int r = 0; r < rounds; ++r) {
    const int i = i_lo + r * nwarps + warp;
    const bool active = i < i_hi;                        // warp-uniform
    const size_t g = ag0 + (active ? i : i_lo);
    const size_t row = g * N + n;
    float qi[8];
    collision_consts(a, g, qi);
    const float rad_i = qi[0], mov_i = qi[3];
    float loss_i = 0.f;
    for (int t0 = 0; t0 < T; t0 += 32) {
      const int t = t0 + lane;
      const bool live = active && t < T;
      float gPx = 0.f, gPy = 0.f, gPsi = 0.f, pen_sum = 0.f;
      // agent i's own pose: from the staged scene, or evaluated here
      float4 pi = make_float4(0.f, 0.f, 0.f, 0.f);
      if (live && a.w_ac != 0.f) pi = one_tile ? reinterpret_cast<const float4*>(pose)[(size_t)i * T + t] : world_pose(a, g, n, t);
      const float Pix = pi.x, Piy = pi.y, ci = pi.z, si = pi.w;
      for (int j0 = 0; j0 < A; j0 += P) {
        const int nt = min(P, A - j0);
        if (!one_tile) {
          __syncthreads();                               // the previous tile is no longer read
          stage_partners(a, pose, agt, ag0 + j0, nt, n, t0, min(32, T - t0), TS);
          __syncthreads();
        }
        if (!live || a.w_ac == 0.f) continue;
        const int tt = one_tile ? t : lane;
        for (int jj = 0; jj < nt; ++jj) {
          if (j0 + jj == i) continue;
          const float* qj = agt + jj * 8;
          const float* pj = pose + ((size_t)jj * TS + tt) * 4;
          float pd = rad_i + qj[0] + a.buffer;
          {
            // the disk centres lie within reach_i / reach_j of the agents' centres: when the centres are further apart than
            // pd + both reaches no pair of disks is within the penalty distance and the pair (i, j) contributes nothing
            const float ddx = Pix - pj[0], ddy = Piy - pj[1];
            const float reach = fmaxf(fabsf(qi[1]), fabsf(qi[2])) + fmaxf(fabsf(qj[1]), fabsf(qj[2]));
            const float lim = (pd + reach) * 1.0001f + 1e-4f;
            if (ddx * ddx + ddy * ddy > lim * lim) continue;
          }
          float best = 3.4e38f, bdx = 0.f, bdy = 0.f, bxi = 0.f;
          for (int d = 0; d < a.D; ++d) {
            float xi = linspace_at(qi[1], qi[2], a.D, d);
            float cx = Pix + xi * ci, cy = Piy + xi * si;
            for (int e = 0; e < a.D; ++e) {
              float xj = linspace_at(qj[1], qj[2], a.D, e);
              float dx = cx - (pj[0] + xj * pj[2]), dy = cy - (pj[1] + xj * pj[3]);
              float dist = sqrtf(dx * dx + dy * dy);
              if (dist < best) { best = dist; bdx = dx; bdy = dy; bxi = xi; }
            }
          }
          if (best <= pd) {
            pen_sum += 1.0f - best / pd;
            if (mov_i != 0.f && best > 0.f) {
              // pair (i,j) is in l_i; pair (j,i) is in l_j when j moves (guidance_loss.py:617-620)
              float f = (1.0f + qj[3]) / (best * pd);
              float gx = -bdx * f, gy = -bdy * f;
              gPx += gx; gPy += gy; gPsi += bxi * (-si * gx + ci * gy);
            }
          }
        }
      }
      if (!live) continue;
      const float wt = wts[t];
      float kk = a.w_ac * inv_AN * (1.0f / (float)A) * wt;
      gPx *= kk; gPy *= kk; gPsi *= kk;
      // back to the agent frame: p = R^T P ; dPsi/dpsi through atan2(R [cos, sin])
      const float* tr = a.traj + (row * T + t) * 6;
      float psi = tr[3], c = cosf(psi), sn = sinf(psi);
      float hx = qi[4] * c + qi[5] * sn, hy = qi[6] * c + qi[7] * sn;
      float dhx = -qi[4] * sn + qi[5] * c, dhy = -qi[6] * sn + qi[7] * c;
      float dPsi_dpsi = (hx * dhy - hy * dhx) / (hx * hx + hy * hy);
      float* o = a.dtraj + (row * T + t) * 4;
      o[0] = qi[4] * gPx + qi[6] * gPy;
      o[1] = qi[5] * gPx + qi[7] * gPy;
      o[2] = 0.f;
      o[3] = gPsi * dPsi_dpsi;
      loss_i += wt * pen_sum;
    }
    if (!active) continue;
#pragma unroll
    for (int o = 16; o; o >>= 1) loss_i += __shfl_xor_sync(0xffffffffu, loss_i, o);
    if (lane == 0 && a.loss) a.loss[row] = (mov_i != 0.f) ? loss_i / (float)A : 0.f;
  }
  __syncthreads();

  if (a.loss)
    for (int i = i_lo + tid; i < i_hi; i += nthr) a.loss[(size_t)a.R + (size_t)(ag0 + i) * N + n] = 0.f;   // map term: own kernel

  // ---------------- target position (softmin-weighted squared distance): warp per agent ------------
  if (a.w_tp != 0.f && a.target) {
    const int t0 = (int)(a.min_target_time * (float)T);
    for (int i = i_lo + warp; i < i_hi; i += nwarps) {
      const size_t g = ag0 + i;
      const size_t row = (size_t)g * N + n;
      // stationary agents were detached in place by the agent-collision term (guidance_loss.py:511-515)
      const bool has_grad = !(a.w_ac != 0.f && !is_moving(a, g));
      const float l = target_pos_term(a.traj + (size_t)row * T * 6, a.dtraj + (size_t)row * T * 4, a.target[g * 2 + 0], a.target[g * 2 + 1], t0, T,
                                      lane, has_grad ? a.w_tp * inv_AN : 0.f);
      if (lane == 0 && a.loss) a.loss[2 * (size_t)a.R + row] = l;
    }
  } else if (a.loss) {
    for (int i = i_lo + tid; i < i_hi; i += nthr) a.loss[2 * (size_t)a.R + (size_t)(ag0 + i) * N + n] = 0.f;
  }
  __syncthreads();       // the waypoint term touches other (row, step) entries of dtraj[..][0..1] than the lanes above

  // ---------------- waypoint terms (SURVEY.md sec. 8 f-4): warp per agent --------------------------------------------
  //   TargetPosAtTimeLoss (guidance_loss.py:630-670), the exact / progress branches of GlobalTargetPosAtTimeLoss (:930-1031) and
  //   GlobalTargetPosLoss (:1033-1135) with compute_progress_loss (:876-927); which branch an agent takes is host logic (wp_mode)
  if (a.w_wp != 0.f && a.wp_mode) {
    for (int i = i_lo + warp; i < i_hi; i += nwarps) {
      const size_t g = ag0 + i;
      const size_t row = (size_t)g * N + n;
      const int mode = a.wp_mode[g];
      const bool has_grad = !(a.w_ac != 0.f && !is_moving(a, g));
      const float kk = has_grad ? a.w_wp * inv_AN * (a.wp_w ? a.wp_w[g] : 1.f) : 0.f;
      const float* tr = a.traj + (size_t)row * T * 6;
      float* dt_ = a.dtraj + (size_t)row * T * 4;
      const float tx = a.wp_target[g * 2 + 0], ty = a.wp_target[g * 2 + 1];
      float l = 0.f;
      if (mode == 4) {
        l = target_pos_term(tr, dt_, tx, ty, (int)(a.min_target_time * (float)T), T, lane, kk);
      } else if (mode != 0 && lane == 0) {
        const int ts = min(max(a.wp_time[g], 0), T - 1);
        const float gd = a.wp_dist[g];
        if (mode == 1) {
          const float dx = tr[ts * 6] - tx, dy = tr[ts * 6 + 1] - ty, d = sqrtf(dx * dx + dy * dy);
          l = d;
          if (d > 0.f) { dt_[ts * 4] += kk * dx / d; dt_[ts * 4 + 1] += kk * dy / d; }
        } else {
          const float ex = tr[(T - 1) * 6] - tx, ey = tr[(T - 1) * 6 + 1] - ty, dl = sqrtf(ex * ex + ey * ey);
          if (mode == 2) {
            l = fmaxf(dl - gd, 0.f);
            if (dl - gd > 0.f && dl > 0.f) { dt_[(T - 1) * 4] += kk * ex / dl; dt_[(T - 1) * 4 + 1] += kk * ey / dl; }
          } else {
            const float fx = tr[0] - tx, fy = tr[1] - ty, df = sqrtf(fx * fx + fy * fy);
            const float e = gd - (df - dl);
            l = fmaxf(e, 0.f);
            if (e > 0.f) {
              if (df > 0.f) { dt_[0] -= kk * fx / df; dt_[1] -= kk * fy / df; }
              if (dl > 0.f) { dt_[(T - 1) * 4] += kk * ex / dl; dt_[(T - 1) * 4 + 1] += kk * ey / dl; }
            }
          }
        }
      }
      if (lane == 0 && a.loss) a.loss[6 * (size_t)a.R + row] = l;
    }
  } else if (a.loss) {
    for (int i = i_lo + tid; i < i_hi; i += nthr) a.loss[6 * (size_t)a.R + (size_t)(ag0 + i) * N + n] = 0.f;
  }
  __syncthreads();       // the terms below add to dtraj[..][2] of the same rows (different lanes <-> steps than above)

  // ---------------- speed / acceleration terms (SURVEY.md sec. 8 f-4): warp per agent, lanes over time -------------------
  //   TargetSpeedLoss (guidance_loss.py:219-254)   mean_t |v_t - v*_t|
  //   AccLimitLoss    (guidance_loss.py:1444-1468)  mean_t max(|acc_t| - limit, 0)   (acc = de-scaled action: gradient goes to dacc)
  //   SpeedLimitLoss  (guidance_loss.py:1509-1538)  mean_t max(|v_t| - limit, 0)
  const bool any_sp = (a.w_ts != 0.f && a.tspeed) || a.w_al != 0.f || a.w_sl != 0.f;
  if (any_sp || a.loss) {
    const float invT = 1.0f / (float)T;
    for (int i = i_lo + warp; i < i_hi; i += nwarps) {
      const size_t g = ag0 + i;
      const size_t row = (size_t)g * N + n;
      const bool has_grad = !(a.w_ac != 0.f && !is_moving(a, g));     // in-place detach of stationary agents, as above
      const float* tr = a.traj + (size_t)row * T * 6;
      float l_ts = 0.f, l_al = 0.f, l_sl = 0.f;
      for (int t = lane; t < T; t += 32) {
        const float v = tr[t * 6 + 2], acc = tr[t * 6 + 4];
        float gv = 0.f, ga = 0.f;
        if (a.w_ts != 0.f && a.tspeed) {
          const float d = v - a.tspeed[(size_t)g * T + t];
          l_ts += fabsf(d);
          gv += a.w_ts * (float)((d > 0.f) - (d < 0.f));
        }
        if (a.w_sl != 0.f) {
          const float e = fabsf(v) - a.speed_limit;
          if (e >= 0.f) { l_sl += e; gv += a.w_sl * (float)((v > 0.f) - (v < 0.f)); }
        }
        if (a.w_al != 0.f) {
          const float e = fabsf(acc) - a.acc_limit;
          if (e >= 0.f) { l_al += e; ga = a.w_al * (float)((acc > 0.f) - (acc < 0.f)); }
        }
        if (any_sp) {
          const float kk = has_grad ? inv_AN * invT : 0.f;
          a.dtraj[((size_t)row * T + t) * 4 + 2] += kk * gv;
          if (a.dacc) a.dacc[(size_t)row * T + t] = kk * ga;
        }
      }
      if (a.loss) {
#pragma unroll
        for (int o = 16; o; o >>= 1) {
          l_ts += __shfl_xor_sync(0xffffffffu, l_ts, o); l_al += __shfl_xor_sync(0xffffffffu, l_al, o); l_sl += __shfl_xor_sync(0xffffffffu, l_sl, o);
        }
        if (lane == 0) {
          a.loss[3 * (size_t)a.R + row] = l_ts * invT; a.loss[4 * (size_t)a.R + row] = l_al * invT; a.loss[5 * (size_t)a.R + row] = l_sl * invT;
        }
      }
    }
  }
}


// ---------------- map collision (MapCollisionLoss.forward, guidance_loss.py:772-870) --------------------------------
// Two kernels.  (1) guidance_map_screen_kernel, one THREAD per (row, step): the raster-space bounding box of the footprint's four
// corners (the sample points are a grid spanned by them, so every sample pixel lies inside it; widened by a pixel fraction against
// rounding) is read from the bit-packed map, a few bytes per pixel row.  All of its pixels drivable: no sample point is off the
// road; none drivable: none is on it; either way loss and gradient are zero (only partially overlapping steps contribute) and
// nothing else is to do.  The other items are appended to a work list.  (2) guidance_map_list_kernel, one WARP per listed item
// (persistent warps striding over the list): the 10 x 10 sample points, their map look-ups and the nearest on-road point of every
// off-road one.
// byte-per-pixel maps -> one bit per pixel (pixel x = bit x & 7 of byte x >> 3, rows of `pitch` bytes): what the screen reads
__global__ void __launch_bounds__(256) guidance_map_pack_kernel(const uint8_t* __restrict__ dmap, int H, int W, int pitch, int n_maps,
                                                                uint8_t* __restrict__ out) {
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)n_maps * H * pitch) return;
  const int bx = (int)(idx % pitch);
  const size_t rowi = idx / pitch;                        // map * H + y
  const uint8_t* src = dmap + rowi * W + (size_t)bx * 8;
  uint32_t v = 0;
  for (int k = 0; k < 8; ++k)
    if (bx * 8 + k < W && src[k] != 0) v |= 1u << k;
  out[idx] = (uint8_t)v;
}

__global__ void __launch_bounds__(256) guidance_map_screen_kernel(LossArgs a) {
  const int T = a.T, N = a.N;
  const int item = blockIdx.x * blockDim.x + threadIdx.x;
  bool flag = false;
  if (item < a.R * T) {
    const int row = item / T, g = row / N;
    if (fabsf(__ldg(a.speed + g)) > a.speed_th) {        // loss and gradient are zero for non-moving agents
      flag = true;
      if (a.pk) {
        const float* M = a.rfa + (size_t)g * 9;
        const float* tr = a.traj + (size_t)item * 6;
        const float L = __ldg(a.extent + g * 3 + 0), Wd = __ldg(a.extent + g * 3 + 1);
        const float px = tr[0], py = tr[1];
        float sn, c;
        sincosf(tr[3], &sn, &c);
        float x0 = 3.4e38f, x1 = -3.4e38f, y0 = 3.4e38f, y1 = -3.4e38f;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float lx = ((k & 1) ? 0.5f : -0.5f) * L, ly = ((k & 2) ? 0.5f : -0.5f) * Wd;
          const float qx = lx * c - ly * sn + px, qy = lx * sn + ly * c + py;
          const float rx = M[0] * qx + M[1] * qy + M[2], ry = M[3] * qx + M[4] * qy + M[5];
          x0 = fminf(x0, rx); x1 = fmaxf(x1, rx); y0 = fminf(y0, ry); y1 = fmaxf(y1, ry);
        }
        // pixel box of the footprint: truncation + clamp as in the sample-point path, widened by 1/16 pixel (+ a relative part for
        // far-away coordinates) so that the rounding of an interior point can never put its pixel outside the box
        const float ex = 0.0625f + 1e-5f * fmaxf(fabsf(x0), fabsf(x1)), ey = 0.0625f + 1e-5f * fmaxf(fabsf(y0), fabsf(y1));
        if (x0 == x0 && x1 == x1 && y0 == y0 && y1 == y1) {           // a NaN pose goes to the full path
          const int cx0 = (int)fminf(fmaxf(floorf(x0 - ex), 0.f), (float)(a.W - 1)), cx1 = (int)fminf(fmaxf(floorf(x1 + ex), 0.f), (float)(a.W - 1));
          const int cy0 = (int)fminf(fmaxf(floorf(y0 - ey), 0.f), (float)(a.H - 1)), cy1 = (int)fminf(fmaxf(floorf(y1 + ey), 0.f), (float)(a.H - 1));
          const int b0 = cx0 >> 3, nb = (cx1 >> 3) - b0 + 1, width = cx1 - cx0 + 1;
          if (nb <= 8 && cy1 - cy0 < 64) {                             // larger boxes (a footprint of > 56 pixels) go to the full path
            // every pixel of the box drivable, or none: n_off is 0 or P and the term vanishes (guidance_loss.py:807-809)
            const uint64_t need = width >= 64 ? ~0ull : ((1ull << width) - 1ull);
            const uint8_t* rowp = a.pk + ((size_t)g * a.H + cy0) * a.pk_pitch + b0;
            bool all_on = true, all_off = true;
            for (int y = cy0; y <= cy1; ++y, rowp += a.pk_pitch) {
              uint64_t v = 0;
              for (int k = 0; k < nb; ++k) v |= (uint64_t)__ldg(rowp + k) << (8 * k);
              v = (v >> (cx0 & 7)) & need;
              all_on = all_on && v == need;
              all_off = all_off && v == 0ull;
            }
            flag = !(all_on || all_off);
          }
        }
      }
    }
    if (a.assign && !flag) reinterpret_cast<float4*>(a.dtraj)[item] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  // warp-aggregated append
  const uint32_t m = __ballot_sync(0xffffffffu, flag);
  if (m) {
    const int lane = threadIdx.x & 31;
    int base = 0;
    if (lane == 0) base = atomicAdd(a.work, __popc(m));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (flag) a.work[2 + base + __popc(m & ((1u << lane) - 1u))] = item;
  }
}

// Nearest on-road sample point of an off-road one.  The sample points are a regular nl x nw grid in the agent frame, so inside a grid
// row the on-road point nearest to column jp is the first set bit at or left of jp or the first one right of it; only those <= 2 nl
// candidates get their distance evaluated -- in the SAME fp32 world-frame arithmetic as the exhaustive search, whose result (minimum,
// argmin, number of exact ties) they reproduce as long as the rounding noise of the coordinates is far below the grid spacing.  When
// it is not (poses thousands of metres from the origin) the warp takes the exhaustive search.
__global__ void __launch_bounds__(256) guidance_map_list_kernel(LossArgs a) {
  __shared__ float qxs[8][128], qys[8][128];
  __shared__ float2 unit_pt[128];                        // (lwise, wwise) of sample point p: no per-point integer division
  __shared__ uchar2 ij_pt[128];                          // (grid row, grid column) of sample point p
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int T = a.T, N = a.N;
  const int nl = a.nl, nw = a.nw, P = nl * nw;
  if (threadIdx.x < 128) {
    const int p = threadIdx.x;
    unit_pt[p] = p < P ? make_float2(a.lwise[p / nw], a.wwise[p % nw]) : make_float2(0.f, 0.f);
    ij_pt[p] = p < P ? make_uchar2((unsigned char)(p / nw), (unsigned char)(p % nw)) : make_uchar2(0, 0);
  }
  __syncthreads();
  const int n_items = *reinterpret_cast<volatile int*>(a.work);
  const int wb = a.packed ? (a.W + 7) >> 3 : a.W;
  const float wmax = (float)a.W, hmax = (float)a.H;
  for (int wi = blockIdx.x * 8 + warp; wi < n_items; wi += gridDim.x * 8) {
    const int item = a.work[2 + wi];
    const int row = item / T, t = item - row * T;
    const int g = row / N;
    // every input of this (row, step) is fetched before the first use: one memory round trip instead of a chain of three
    const float* M = a.rfa + (size_t)g * 9;
    const float* tr = a.traj + (size_t)item * 6;
    const float L = __ldg(a.extent + g * 3 + 0), Wd = __ldg(a.extent + g * 3 + 1);
    const float m0 = __ldg(M + 0), m1 = __ldg(M + 1), m2 = __ldg(M + 2), m3 = __ldg(M + 3), m4 = __ldg(M + 4), m5 = __ldg(M + 5);
    const float2 pxy = *reinterpret_cast<const float2*>(tr);
    const float px = pxy.x, py = pxy.y, psi = tr[3];
    const uint8_t* dm = a.dmap + (size_t)g * a.H * wb;
    float sn, c;
    sincosf(psi, &sn, &c);
    uint32_t offm[4];
    int n_off = 0;
    __syncwarp();                                         // the previous item's reads of qxs / qys are complete
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      int p = lane + 32 * q;
      bool off = false;
      if (p < P) {
        const float2 up = unit_pt[p];
        float lx = up.x * L, ly = up.y * Wd;
        float qx = lx * c - ly * sn + px, qy = lx * sn + ly * c + py;
        qxs[warp][p] = qx; qys[warp][p] = qy;
        float rx = m0 * qx + m1 * qy + m2, ry = m3 * qx + m4 * qy + m5;
        // .long() truncates (guidance_loss.py:796), then clamp to the raster; done in fp32 -> int32 (identical on [-1, W])
        int cx = (int)fminf(fmaxf(rx, -1.f), wmax), cy = (int)fminf(fmaxf(ry, -1.f), hmax);
        cx = cx < 0 ? 0 : (cx > a.W - 1 ? a.W - 1 : cx);
        cy = cy < 0 ? 0 : (cy > a.H - 1 ? a.H - 1 : cy);
        off = a.packed ? ((dm[cy * wb + (cx >> 3)] >> (cx & 7)) & 1) == 0 : dm[cy * wb + cx] == 0;
      }
      offm[q] = __ballot_sync(0xffffffffu, off);
      n_off += __popc(offm[q]);
    }
    float gx = 0.f, gy = 0.f, gpsi = 0.f, lsum = 0.f;
    if (n_off != 0 && n_off != P) {                       // only partially overlapping steps contribute
      __syncwarp();
      const float diag = sqrtf(L * L + Wd * Wd);
      // on-road bits of the warp's points, per 32-point word
      uint32_t onm[4];
#pragma unroll
      for (int w = 0; w < 4; ++w) {
        const int left = P - w * 32;
        onm[w] = ~offm[w] & (left >= 32 ? 0xffffffffu : (left > 0 ? ((1u << left) - 1u) : 0u));
      }
      // lane i < nl: the on-road bits of grid row i (columns 0 .. nw - 1)
      uint32_t rowmask = 0;
      if (lane < nl) {
        const int start = lane * nw, w = start >> 5, sh = start & 31;
        const uint32_t lo = w == 0 ? onm[0] : w == 1 ? onm[1] : w == 2 ? onm[2] : onm[3];
        const uint32_t hi = w == 0 ? onm[1] : w == 1 ? onm[2] : w == 2 ? onm[3] : 0u;
        rowmask = ((lo >> sh) | (sh ? hi << (32 - sh) : 0u)) & ((1u << nw) - 1u);
      }
      // rounding noise of the coordinates vs the grid spacing (see the comment above the kernel)
      const float sl = nl > 1 ? L / (float)(nl - 1) : 3.4e38f, sw = nw > 1 ? Wd / (float)(nw - 1) : 3.4e38f, smin = fminf(sl, sw);
      const bool pruned = !a.exhaustive && 6.f * diag * 2.5e-7f * (fabsf(px) + fabsf(py) + L + Wd) < 0.5f * smin * smin;
      const int c0 = __popc(offm[0]), c1 = c0 + __popc(offm[1]), c2 = c1 + __popc(offm[2]);
      // the off-road points are dealt to the lanes in order: pass k takes the 32 k-th .. (32 k + 31)-th of them
      for (int r0 = 0; r0 < n_off; r0 += 32) {
        const int r = r0 + lane;
        const bool active = r < n_off;
        int p = 0;
        if (active) {
          const int w = r < c0 ? 0 : r < c1 ? 1 : r < c2 ? 2 : 3;
          const int base = w == 0 ? 0 : w == 1 ? c0 : w == 2 ? c1 : c2;
          const uint32_t m = w == 0 ? offm[0] : w == 1 ? offm[1] : w == 2 ? offm[2] : offm[3];
          p = w * 32 + (int)__fns(m, 0, r - base + 1);
        }
        const float pxw = qxs[warp][p], pyw = qys[warp][p];
        float best2 = 3.4e38f, bx = 0.f, by = 0.f;
        int cnt = 0;
        auto consider = [&](int k) {
          const float qx = qxs[warp][k], qy = qys[warp][k];
          const float dx = qx - pxw, dy = qy - pyw;
          const float d2 = dx * dx + dy * dy;
          if (d2 < best2) { best2 = d2; bx = qx; by = qy; cnt = 1; }
          else if (d2 == best2) ++cnt;
        };
        if (pruned) {
          const int jp = ij_pt[p].y;
          for (int i = 0; i < nl; ++i) {
            const uint32_t Mi = __shfl_sync(0xffffffffu, rowmask, i);
            if (!Mi || !active) continue;
            const uint32_t le = Mi & ((2u << jp) - 1u), gt = (Mi >> jp) >> 1;
            if (le) consider(i * nw + 31 - __clz(le));
            if (gt) consider(i * nw + jp + __ffs(gt));
          }
        } else if (active) {
#pragma unroll 1
          for (int w = 0; w < 4; ++w) {
            uint32_t on = onm[w];
            while (on) {
              const int k = w * 32 + __ffs(on) - 1;
              on &= on - 1;
              consider(k);
            }
          }
        }
        if (!active) continue;
        const float best = sqrtf(best2);
        lsum += 1.0f - best / diag;
        if (best > 0.f) {
          if (cnt == 1) {
            float f = -1.0f / (best * diag);
            float ggx = (bx - pxw) * f, ggy = (by - pyw) * f;
            gx += ggx; gy += ggy;
            gpsi += ggx * (-(by - py)) + ggy * (bx - px);
          } else {
            // torch.amin splits the gradient evenly over tied minima
            float f = -1.0f / (best * diag * (float)cnt);
            for (int k = 0; k < P; ++k) {
              if ((offm[k >> 5] >> (k & 31)) & 1u) continue;
              float dx = qxs[warp][k] - pxw, dy = qys[warp][k] - pyw;
              if (dx * dx + dy * dy == best2) {
                float ggx = dx * f, ggy = dy * f;
                gx += ggx; gy += ggy;
                gpsi += ggx * (-(qys[warp][k] - py)) + ggy * (qxs[warp][k] - px);
              }
            }
          }
        }
      }
#pragma unroll
      for (int o = 16; o; o >>= 1) {
        gx += __shfl_xor_sync(0xffffffffu, gx, o);
        gy += __shfl_xor_sync(0xffffffffu, gy, o);
        gpsi += __shfl_xor_sync(0xffffffffu, gpsi, o);
        lsum += __shfl_xor_sync(0xffffffffu, lsum, o);
      }
    }
    if (lane == 0) {
      const float wt = a.wts[t];
      float kk = a.w_mc * (1.0f / (float)(a.A * N)) * wt;
      float4* o = reinterpret_cast<float4*>(a.dtraj) + item;
      if (a.assign) {
        *o = make_float4(kk * gx, kk * gy, 0.f, kk * gpsi);
      } else if (n_off != 0 && n_off != P) {
        float4 v = *o;
        v.x += kk * gx; v.y += kk * gy; v.w += kk * gpsi;
        *o = v;
        if (a.loss) atomicAdd(&a.loss[(size_t)a.R + row], wt * lsum);
      }
    }
  }
  // the last CTA to finish resets the list for the next step
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(a.work + 1, 1) == (int)gridDim.x - 1) { a.work[0] = 0; a.work[1] = 0; __threadfence(); }
  }
}

static float host_linspace(float lo, float hi, int n, int i) {
  if (n == 1) return lo;
  float step = (hi - lo) / (float)(n - 1);
  return (i < n / 2) ? lo + step * (float)i : hi - step * (float)(n - 1 - i);
}

int guidance_prepare_maps(CldHandle* h, const CldScene* sc, cudaStream_t s) {
  h->screen_src = nullptr;
  if (!sc || !sc->drivable_map || sc->map_w < 1 || sc->map_h < 1) return 0;     // no screen: every moving item takes the full path
  const int n_maps = sc->num_scenes * sc->agents_per_scene;
  if (sc->map_packed) {
    h->screen_pk = sc->drivable_map; h->screen_pitch = (sc->map_w + 7) / 8;
  } else {
    const int pitch = (sc->map_w + 7) / 8;
    const size_t bytes = (size_t)n_maps * sc->map_h * pitch;
    if (bytes > h->map_bits_bytes) {
      // grows only when a larger scene / map arrives (first guided call): not on the per-step path
      uint8_t* p = nullptr;
      CLD_CUDA_OK(h, cudaMalloc((void**)&p, bytes));
      h->allocs.push_back(p);
      h->map_bits = p; h->map_bits_bytes = bytes;
    }
    guidance_map_pack_kernel<<<(unsigned)((bytes + 255) / 256), 256, 0, s>>>(sc->drivable_map, sc->map_h, sc->map_w, pitch, n_maps, h->map_bits);
    CLD_LAUNCH_OK(h, "guidance_map_pack_kernel");
    h->screen_pk = h->map_bits; h->screen_pitch = pitch;
  }
  h->screen_src = sc->drivable_map; h->screen_agents = n_maps; h->screen_h = sc->map_h; h->screen_w = sc->map_w; h->screen_packed = sc->map_packed;
  return 0;
}

static int launch_map(CldHandle* h, const LossArgs& a, cudaStream_t s) {
  const int items = a.R * a.T;
  guidance_map_screen_kernel<<<(items + 255) / 256, 256, 0, s>>>(a);
  CLD_LAUNCH_OK(h, "guidance_map_screen_kernel");
  if (h->env_map_stats) {                       // debug (CLD_MAP_STATS=1): how many items the screen lets through
    int n = 0;
    CLD_CUDA_OK(h, cudaStreamSynchronize(s));
    CLD_CUDA_OK(h, cudaMemcpy(&n, a.work, sizeof(int), cudaMemcpyDeviceToHost));
    fprintf(stderr, "[map screen] %d of %d (row, step) items listed\n", n, items);
  }
  // persistent warps over the list: 8 CTAs of 8 warps per SM at most, no more warps than items could ever be listed
  int grid = h->num_sms * 8;
  if (grid * 8 > items) grid = (items + 7) / 8;
  guidance_map_list_kernel<<<grid, 256, 0, s>>>(a);
  CLD_LAUNCH_OK(h, "guidance_map_list_kernel");
  return 0;
}

int guidance_loss_grad(CldHandle* h, const float* traj, const CldScene* sc, const CldGuidanceConfig* g, float* dtraj,
                       float* dtraj_map, float* dacc, float* loss, int R, cudaStream_t s) {
  if (!sc || !g) return fail(h, CLD_ERR_ARG, "scene / guidance config missing");
  int rc;
  const int S = sc->num_scenes, A = sc->agents_per_scene, N = sc->num_samp, T = h->cfg.horizon;
  if (R != S * A * N) return fail(h, CLD_ERR_ARG, "R=%d does not match S*A*N=%d*%d*%d", R, S, A, N);
  if (A < 1) return fail(h, CLD_ERR_UNSUPPORTED, "agents_per_scene must be >= 1");
  if (g->num_disks < 1 || g->num_disks > 5) return fail(h, CLD_ERR_UNSUPPORTED, "num_disks must be in [1,5]");
  if (g->num_points_l < 1 || g->num_points_l > 16 || g->num_points_w < 1 || g->num_points_w > 16 ||
      g->num_points_l * g->num_points_w > 128)
    return fail(h, CLD_ERR_UNSUPPORTED, "num_points_lw must be <=16 each and <=128 points in total");
  if (!sc->extent || !sc->world_from_agent || !sc->curr_speed) return fail(h, CLD_ERR_ARG, "scene tensors missing");
  if (g->w_map_collision != 0.f && (!sc->drivable_map || !sc->raster_from_agent))
    return fail(h, CLD_ERR_ARG, "map_collision needs drivable_map and raster_from_agent");
  LossArgs a;
  a.traj = traj; a.dtraj = dtraj; a.loss = loss;
  a.extent = sc->extent; a.wfa = sc->world_from_agent; a.rfa = sc->raster_from_agent; a.speed = sc->curr_speed;
  a.target = sc->target_pos; a.dmap = sc->drivable_map; a.H = sc->map_h; a.W = sc->map_w; a.packed = sc->map_packed;
  a.S = S; a.A = A; a.N = N; a.T = T; a.R = R;
  a.w_ac = g->w_agent_collision; a.w_mc = g->w_map_collision; a.w_tp = g->w_target_pos;
  a.tspeed = sc->target_speed; a.w_ts = g->w_target_speed; a.w_al = g->w_acc_limit; a.acc_limit = g->acc_limit;
  a.w_sl = g->w_speed_limit; a.speed_limit = g->speed_limit; a.dacc = a.w_al != 0.f ? dacc : nullptr;
  a.w_wp = g->w_waypoint; a.wp_target = sc->wp_target; a.wp_mode = sc->wp_mode; a.wp_time = sc->wp_time; a.wp_dist = sc->wp_dist; a.wp_w = sc->wp_weight;
  if (a.w_wp != 0.f && (!sc->wp_target || !sc->wp_mode || !sc->wp_time || !sc->wp_dist))
    return fail(h, CLD_ERR_ARG, "waypoint guidance needs CldScene.wp_target / wp_mode / wp_time / wp_dist");
  if (a.w_ts != 0.f && !sc->target_speed) return fail(h, CLD_ERR_ARG, "target_speed guidance needs CldScene.target_speed");
  if (a.w_al != 0.f && !dacc) return fail(h, CLD_ERR_STATE, "internal: acc-limit guidance without a d(acc) buffer");
  a.work = h->map_work; a.assign = 0; a.exhaustive = h->env_map_exhaustive ? 1 : 0;
  // the screen data belongs to the maps guidance_prepare_maps last saw
  const bool screen_ok = h->screen_src == (const void*)sc->drivable_map && h->screen_agents >= S * A && h->screen_h == sc->map_h &&
                         h->screen_w == sc->map_w && h->screen_packed == sc->map_packed;
  a.pk = screen_ok ? h->screen_pk : nullptr; a.pk_pitch = h->screen_pitch;
  a.D = g->num_disks; a.buffer = g->buffer_dist; a.decay = g->decay_rate; a.speed_th = g->speed_th;
  a.min_target_time = g->min_target_time; a.nl = g->num_points_l; a.nw = g->num_points_w;
  for (int i = 0; i < 16; ++i) {
    a.lwise[i] = i < a.nl ? host_linspace(-0.5f, 0.5f, a.nl, i) : 0.f;
    a.wwise[i] = i < a.nw ? host_linspace(-0.5f, 0.5f, a.nw, i) : 0.f;
  }
  {
    // exp_weights: python-double powers cast to fp32, fp32 sum, fp32 divide (guidance_loss.py:607-608)
    float sum = 0.f;
    for (int t = 0; t < T; ++t) { a.wts[t] = (float)pow((double)g->decay_rate, (double)t); sum += a.wts[t]; }
    for (int t = 0; t < T; ++t) a.wts[t] /= sum;
    for (int t = T; t < CLD_MAX_T; ++t) a.wts[t] = 0.f;
  }
  // the whole scene (at most 133 KB: A = 64, T = 128), or one tile of partners (65 KB and the decay weights)
  const bool one_tile = A <= SCENE_TILE;
  const size_t smem = ((size_t)(one_tile ? A : PARTNER_TILE) * ((one_tile ? T : 32) * 4 + 8) + T) * sizeof(float);
  CLD_CUDA_OK(h, cudaFuncSetAttribute(guidance_loss_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const bool fork = dtraj_map != nullptr && loss == nullptr && a.w_mc != 0.f;
  if (fork) {
    // the two loss kernels are independent given the trajectories: the map-collision kernel runs on the auxiliary stream into
    // its own (zeroed) gradient buffer while the agent-collision kernel runs here
    if (!h->aux_stream) {
      CLD_CUDA_OK(h, cudaStreamCreateWithFlags(&h->aux_stream, cudaStreamNonBlocking));
      CLD_CUDA_OK(h, cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
      CLD_CUDA_OK(h, cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    }
    CLD_CUDA_OK(h, cudaEventRecord(h->ev_fork, s));
    CLD_CUDA_OK(h, cudaStreamWaitEvent(h->aux_stream, h->ev_fork, 0));
    LossArgs am = a;
    am.dtraj = dtraj_map; am.assign = 1;              // the two map kernels write every item of their own buffer
    if ((rc = launch_map(h, am, h->aux_stream))) return rc;
    CLD_CUDA_OK(h, cudaEventRecord(h->ev_join, h->aux_stream));
  }
  // enough CTAs for ~2 per SM: the agents of a scene are split over gridDim.y CTAs when there are few (scene, sample) pairs
  int split = 1;
  if (one_tile) {
    while (S * N * split < 2 * h->num_sms && split * 2 <= (A + 3) / 4) split *= 2;
  } else {
    // several tiles: at most one agent per warp (16 per CTA), so a CTA stages each tile once; down to 4 agents per CTA while
    // the grid is short of 2 CTAs per SM
    int per = 16;
    while (per > 4 && (size_t)S * N * ((A + per - 1) / per) < 2 * (size_t)h->num_sms) per /= 2;
    split = (A + per - 1) / per;
  }
  const int per_cta = (A + split - 1) / split;
  const int threads = 32 * (per_cta < 4 ? 4 : (per_cta > 16 ? 16 : per_cta));       // one warp per agent, 4 .. 16 warps
  guidance_loss_grad_kernel<<<dim3((unsigned)(S * N), (unsigned)split), threads, smem, s>>>(a);
  CLD_LAUNCH_OK(h, "guidance_loss_grad_kernel");
  if (fork) {
    CLD_CUDA_OK(h, cudaStreamWaitEvent(s, h->ev_join, 0));
  } else if (a.w_mc != 0.f) {
    if ((rc = launch_map(h, a, s))) return rc;
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// backward: d(traj) -> d(scaled actions) -> BPTT -> dz -> optimizer step
// ------------------------------------------------------------------------------------------------
struct BwdArgs {
  const float *z_mean, *act, *curr, *dtraj, *stash;
  const float *wih0, *whh0, *wih1, *whh1, *h2a_w;   // original [4H][in] layouts
  float *z_out, *grad_out;
  int R, T;
  float dt, acce_lo, acce_hi, v_lo, v_hi, max_steer, max_yawvel, a_mean, a_std, w_mean, w_std;
  int optimizer; float lr;
};

// reverse of unicycle_row for one row (SURVEY.md Appendix C); writes d(scaled action) [T][2]
__device__ void unicycle_row_backward(const float* act, const float* curr, const float* dtr, int T, const BwdArgs& a,
                                      float* scr /*[4][T+1]*/, float* dact) {
  float* sk = scr;                 // raw cumulative speed s_k, k=0..T
  float* psik = scr + (T + 1);     // yaw psi_k, k=0..T
  float* vbar = scr + 2 * (T + 1); // k=0..T-1
  float* msk = scr + 3 * (T + 1);  // bit0: acc clip passes, bit1: yaw-rate clip passes
  float s = curr[2], psi = curr[3];
  float vprev = clipg(s, a.v_lo, a.v_hi);
  sk[0] = s; psik[0] = psi;
  for (int k = 0; k < T; ++k) {
    float a_raw = __fadd_rn(__fmul_rn(act[k * 2 + 0], a.a_std), a.a_mean);
    float w_raw = __fadd_rn(__fmul_rn(act[k * 2 + 1], a.w_std), a.w_mean);
    float ac = clipg(a_raw, a.acce_lo, a.acce_hi);
    s = __fadd_rn(s, __fmul_rn(ac, a.dt));
    float vnext = clipg(s, a.v_lo, a.v_hi);
    vbar[k] = __fmul_rn(0.5f, __fadd_rn(vprev, vnext));
    float ve = fabsf(vprev);
    float yb = fmaxf(fminf(__fmul_rn(a.max_steer, ve), __fdiv_rn(a.max_yawvel, fmaxf(ve, 0.1f))), 0.1f);
    float w = clipg(w_raw, -yb, yb);
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
    dact[m * 2 + 0] = a.a_std * du0;
    dact[m * 2 + 1] = a.w_std * du1;
    dvbar_next = dvbar; direct_next = direct;
  }
}

template <int RB>
__global__ void __launch_bounds__(256, 1) lstm_backward_update_kernel(BwdArgs a) {
  constexpr int H = 64, PPT = RB * H / 256;
  extern __shared__ __align__(16) float sm[];
  const int T = a.T, R = a.R;
  float* acts = sm;                                  // [RB][T][2]
  float* dtr = acts + RB * T * 2;                    // [RB][T][4]
  float* dact = dtr + RB * T * 4;                    // [RB][T][2]
  float* scr = dact + RB * T * 2;                    // [RB][4][T+1]
  float* dh0seq = scr + RB * 4 * (T + 1);            // [T][RB][H]
  float* dzb = dh0seq + (size_t)T * RB * H;          // [RB][256] gate pre-activation grads
  float* part = dzb + RB * 256;                      // [4][RB][H] partial transposed mat-vecs
  float* dhrec = part + 4 * RB * H;                  // [RB][H]
  float* dzout = dhrec + RB * H;                     // [RB][T][4]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, row0 = blockIdx.x * RB;

  for (int i = tid; i < RB * T * 2; i += 256) {
    int b = i / (T * 2);
    acts[i] = (row0 + b < R) ? a.act[(size_t)row0 * T * 2 + i] : 0.f;
  }
  for (int i = tid; i < RB * T * 4; i += 256) {
    int b = i / (T * 4);
    dtr[i] = (row0 + b < R) ? a.dtraj[(size_t)row0 * T * 4 + i] : 0.f;
  }
  __syncthreads();
  if (tid < RB) {
    float cs[4] = {0.f, 0.f, 0.f, 0.f};
    if (row0 + tid < R)
      for (int i = 0; i < 4; ++i) cs[i] = a.curr[(size_t)(row0 + tid) * 4 + i];
    unicycle_row_backward(acts + tid * T * 2, cs, dtr + tid * T * 4, T, a, scr + tid * 4 * (T + 1), dact + tid * T * 2);
  }
  for (int p = tid; p < RB * H; p += 256) dhrec[p] = 0.f;
  __syncthreads();

  // ------------------------------ layer 1 (top) -------------------------------------------------
  {
    const int which = tid >> 7, jh = (tid >> 6) & 1, k = tid & 63;
    const float* Wsrc = which ? a.wih1 : a.whh1;
    float w[128];
#pragma unroll
    for (int jj = 0; jj < 128; ++jj) w[jj] = Wsrc[(size_t)(jh * 128 + jj) * H + k];
    float dcrec[PPT];
#pragma unroll
    for (int i = 0; i < PPT; ++i) dcrec[i] = 0.f;
    const float* st1 = a.stash + (size_t)T * R * 5 * H;
    for (int t = T - 1; t >= 0; --t) {
#pragma unroll
      for (int i = 0; i < PPT; ++i) {
        int p = tid + i * 256, b = p >> 6, u = p & 63;
        float dz_i = 0.f, dz_f = 0.f, dz_g = 0.f, dz_o = 0.f;
        if (row0 + b < R) {
          const float* st = st1 + ((size_t)t * R + row0 + b) * (5 * H) + u;
          float ig = st[0], fg = st[H], gg = st[2 * H], og = st[3 * H], c = st[4 * H];
          float cprev = (t > 0) ? *(st + 4 * H - (ptrdiff_t)R * 5 * H) : 0.f;
          float dh = a.h2a_w[u] * dact[(b * T + t) * 2] + a.h2a_w[H + u] * dact[(b * T + t) * 2 + 1] + dhrec[b * H + u];
          float tc = tanhf(c);
          float dc = dcrec[i] + dh * og * (1.f - tc * tc);
          dz_i = dc * gg * ig * (1.f - ig);
          dz_f = dc * cprev * fg * (1.f - fg);
          dz_g = dc * ig * (1.f - gg * gg);
          dz_o = dh * tc * og * (1.f - og);
          dcrec[i] = dc * fg;
        }
        float* d = dzb + b * 256 + u;
        d[0] = dz_i; d[64] = dz_f; d[128] = dz_g; d[192] = dz_o;
      }
      __syncthreads();
      float acc[RB];
#pragma unroll
      for (int b = 0; b < RB; ++b) acc[b] = 0.f;
#pragma unroll
      for (int j4 = 0; j4 < 32; ++j4) {
#pragma unroll
        for (int b = 0; b < RB; ++b) {
          float4 dv = *reinterpret_cast<const float4*>(dzb + b * 256 + jh * 128 + j4 * 4);
          acc[b] = fmaf(w[j4 * 4 + 0], dv.x, acc[b]); acc[b] = fmaf(w[j4 * 4 + 1], dv.y, acc[b]);
          acc[b] = fmaf(w[j4 * 4 + 2], dv.z, acc[b]); acc[b] = fmaf(w[j4 * 4 + 3], dv.w, acc[b]);
        }
      }
#pragma unroll
      for (int b = 0; b < RB; ++b) part[((which * 2 + jh) * RB + b) * H + k] = acc[b];
      __syncthreads();
      for (int p = tid; p < RB * H; p += 256) {
        dhrec[p] = part[p] + part[RB * H + p];
        dh0seq[(size_t)t * RB * H + p] = part[2 * RB * H + p] + part[3 * RB * H + p];
      }
      __syncthreads();
    }
  }
  // ------------------------------ layer 0 --------------------------------------------------------
  {
    for (int p = tid; p < RB * H; p += 256) dhrec[p] = 0.f;
    __syncthreads();
    const int jq = tid >> 6, k = tid & 63;
    float w[64];
#pragma unroll
    for (int jj = 0; jj < 64; ++jj) w[jj] = a.whh0[(size_t)(jq * 64 + jj) * H + k];
    float4 wi[8];   // weight_ih_l0 rows j = lane*8 .. lane*8+7 (for dz = W_ih^T dgates)
#pragma unroll
    for (int jj = 0; jj < 8; ++jj) wi[jj] = *reinterpret_cast<const float4*>(a.wih0 + (size_t)(lane * 8 + jj) * 4);
    float dcrec[PPT];
#pragma unroll
    for (int i = 0; i < PPT; ++i) dcrec[i] = 0.f;
    const float* st0 = a.stash;
    for (int t = T - 1; t >= 0; --t) {
#pragma unroll
      for (int i = 0; i < PPT; ++i) {
        int p = tid + i * 256, b = p >> 6, u = p & 63;
        float dz_i = 0.f, dz_f = 0.f, dz_g = 0.f, dz_o = 0.f;
        if (row0 + b < R) {
          const float* st = st0 + ((size_t)t * R + row0 + b) * (5 * H) + u;
          float ig = st[0], fg = st[H], gg = st[2 * H], og = st[3 * H], c = st[4 * H];
          float cprev = (t > 0) ? *(st + 4 * H - (ptrdiff_t)R * 5 * H) : 0.f;
          float dh = dh0seq[(size_t)t * RB * H + p] + dhrec[p];
          float tc = tanhf(c);
          float dc = dcrec[i] + dh * og * (1.f - tc * tc);
          dz_i = dc * gg * ig * (1.f - ig);
          dz_f = dc * cprev * fg * (1.f - fg);
          dz_g = dc * ig * (1.f - gg * gg);
          dz_o = dh * tc * og * (1.f - og);
          dcrec[i] = dc * fg;
        }
        float* d = dzb + b * 256 + u;
        d[0] = dz_i; d[64] = dz_f; d[128] = dz_g; d[192] = dz_o;
      }
      __syncthreads();
      float acc[RB];
#pragma unroll
      for (int b = 0; b < RB; ++b) acc[b] = 0.f;
#pragma unroll
      for (int j4 = 0; j4 < 16; ++j4) {
#pragma unroll
        for (int b = 0; b < RB; ++b) {
          float4 dv = *reinterpret_cast<const float4*>(dzb + b * 256 + jq * 64 + j4 * 4);
          acc[b] = fmaf(w[j4 * 4 + 0], dv.x, acc[b]); acc[b] = fmaf(w[j4 * 4 + 1], dv.y, acc[b]);
          acc[b] = fmaf(w[j4 * 4 + 2], dv.z, acc[b]); acc[b] = fmaf(w[j4 * 4 + 3], dv.w, acc[b]);
        }
      }
#pragma unroll
      for (int b = 0; b < RB; ++b) part[(jq * RB + b) * H + k] = acc[b];
      // dz_t = W_ih_l0^T dgates : warp b handles row b (RB <= 8 warps)
      if (warp < RB) {
        float4 s4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
          float dv = dzb[warp * 256 + lane * 8 + jj];
          s4.x = fmaf(wi[jj].x, dv, s4.x); s4.y = fmaf(wi[jj].y, dv, s4.y);
          s4.z = fmaf(wi[jj].z, dv, s4.z); s4.w = fmaf(wi[jj].w, dv, s4.w);
        }
#pragma unroll
        for (int o = 16; o; o >>= 1) {
          s4.x += __shfl_xor_sync(0xffffffffu, s4.x, o); s4.y += __shfl_xor_sync(0xffffffffu, s4.y, o);
          s4.z += __shfl_xor_sync(0xffffffffu, s4.z, o); s4.w += __shfl_xor_sync(0xffffffffu, s4.w, o);
        }
        if (lane == 0) *reinterpret_cast<float4*>(dzout + (warp * T + t) * 4) = s4;
      }
      __syncthreads();
      for (int p = tid; p < RB * H; p += 256)
        dhrec[p] = part[p] + part[RB * H + p] + part[2 * RB * H + p] + part[3 * RB * H + p];
      __syncthreads();
    }
  }
  // ------------------------------ optimizer step (guidance_loss.py:2250-2278) --------------------
  for (int i = tid; i < RB * T * 4; i += 256) {
    int b = i / (T * 4);
    if (row0 + b >= R) continue;
    size_t gi = (size_t)row0 * T * 4 + i;
    float g = dzout[i], z = a.z_mean[gi], zn;
    if (a.optimizer == CLD_OPT_ADAM) {
      // first torch.optim.Adam step: m = 0.1 g, v = 0.001 g^2, bias corrections 0.1 / 0.001, eps 1e-8
      float m = 0.1f * g;
      float v = (0.001f * g) * g;
      float denom = sqrtf(v) / 0.03162277660168379f + 1e-8f;
      float step = a.lr / 0.1f;
      zn = z - step * (m / denom);
    } else {
      zn = z - a.lr * g;
    }
    a.z_out[gi] = zn;
    if (a.grad_out) a.grad_out[gi] = g;
  }
}

template <int RB>
static size_t bwd_smem_bytes(int T) {
  size_t f = (size_t)RB * T * 2 + (size_t)RB * T * 4 + (size_t)RB * T * 2 + (size_t)RB * 4 * (T + 1) +
             (size_t)T * RB * 64 + (size_t)RB * 256 + 4 * (size_t)RB * 64 + (size_t)RB * 64 + (size_t)RB * T * 4;
  return f * sizeof(float);
}

template <int RB>
static int launch_bwd(CldHandle* h, const BwdArgs& a, cudaStream_t s) {
  size_t smem = bwd_smem_bytes<RB>(a.T);
  auto kern = lstm_backward_update_kernel<RB>;
  CLD_CUDA_OK(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<(a.R + RB - 1) / RB, 256, smem, s>>>(a);
  CLD_LAUNCH_OK(h, "lstm_backward_update_kernel");
  return 0;
}

int decode_backward_update(CldHandle* h, const float* z_mean, const float* act, const float* curr, const float* dtraj,
                           const CldGuidanceConfig* g, float* z_out, float* grad_out, int R, cudaStream_t s) {
  const CldConfig& c = h->cfg;
  BwdArgs a;
  a.z_mean = z_mean; a.act = act; a.curr = curr; a.dtraj = dtraj; a.stash = h->stash;
  a.wih0 = h->dec.wih0_raw; a.whh0 = h->dec.whh0_raw; a.wih1 = h->dec.wih1_raw; a.whh1 = h->dec.whh1_raw;
  a.h2a_w = h->dec.h2a_w;
  a.z_out = z_out; a.grad_out = grad_out; a.R = R; a.T = c.horizon;
  a.dt = c.dt; a.acce_lo = c.acce_lo; a.acce_hi = c.acce_hi; a.v_lo = c.v_lo; a.v_hi = c.v_hi;
  a.max_steer = c.max_steer; a.max_yawvel = c.max_yawvel;
  a.a_mean = c.norm_mean[4]; a.a_std = c.norm_std[4]; a.w_mean = c.norm_mean[5]; a.w_std = c.norm_std[5];
  a.optimizer = g->optimizer; a.lr = g->lr;
  if (a.T <= 64) return launch_bwd<8>(h, a, s);
  return launch_bwd<4>(h, a, s);
}

}  // namespace cld
