// SURVEY.md sec. 8 f-2: the PPO inner loop's denoiser update (reference src/trainers/guide_dm_trainer.py:127-183,
// models/dm/dm_model.py:165-174) without autograd: forward of TemporalMapUnet (src/tbsim/models/temporal.py:122-180) that keeps
// what the backward needs, the analytic backward of every layer down to the 148 parameter gradients (written in the state-dict
// layouts the reference's optimizer sees), the PPO clipped-surrogate and MSE loss heads, and Adam (torch.optim.Adam semantics,
// guide_dm_trainer.py:59-65).  fp32 on the CUDA cores: this is the parity-first build of the row (1e-4 against autograd of the real
// reference module); the minibatch is 128 rows (config.yaml:168), i.e. launch- and latency-bound.
//
// Layout: activations channels-last [R, T', C] fp32 as in kernels_unet_fp32.cu.  Every convolution (forward), its data gradient
// and its weight gradient is one implicit GEMM over M = R * T' rows:
//   forward   out[r, j*os+oo, :]  = bias + sum_tap in[r, j*is+io[tap], :] @ W[tap]              (W packed [tap][cin][cout])
//   data grad dIn[r, ti, :]      += sum_tap dOut[r, ...] @ W[tap]^T                              (same kernel, B read transposed)
//   weight    dW[tap][ci][co]     = sum_{r,j} in[r, j*is+io[tap], ci] * dOut[r, j*os+oo, co]     (split over M, fixed-order reduce)
// No atomics anywhere: all reductions have a fixed order, so a step is bit-reproducible.
#include "common.cuh"

namespace cld {

// ------------------------------------------------------------------------------------------------
// implicit GEMM, forward / data gradient
// ------------------------------------------------------------------------------------------------
struct TGemm {
  const float* in0; int c0;     // A source [R, Tin, c0]
  const float* in1; int c1;     // optional concatenated source [R, Tin, c1]
  int Tin;
  const float* w[5];            // per GEMM tap: TRANSB = 0: [K][ldw] (n contiguous);  TRANSB = 1: [N][ldw] (k contiguous)
  int ldw;
  const float* bias;            // [N] or nullptr
  float* out; int Tout; int cout;
  int ntaps; int ioff[5]; int istride, ostride, ooff;
  int Tj; int R; int accum;
};

constexpr int GBN = 64, GBK = 16;

// BM = 128 | 64 | 32 GEMM rows per CTA (256 threads, thread tile BM/16 x 4): a 128-row minibatch gives M = 1 664 .. 6 656 rows, i.e.
// 13 .. 52 tiles of 128 -- the smaller tiles are what fills 148 SMs
template <bool TRANSB, int BM>
__global__ void __launch_bounds__(256) tgemm_kernel(TGemm a) {
  constexpr int RPT = BM / 16;                       // rows per thread
  constexpr int ALOADS = (BM * 4 + 255) / 256;       // float4 loads of the A tile per thread
  __shared__ __align__(16) float As[GBK][BM + 4];
  __shared__ __align__(16) float Bs[GBK][GBN + 4];
  const int tid = threadIdx.x;
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * GBN;
  const int M = a.R * a.Tj;
  const int cin = a.c0 + a.c1;
  const int ty = tid >> 4, tx = tid & 15;
  float acc[RPT][4];
#pragma unroll
  for (int i = 0; i < RPT; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  int a_row[ALOADS], a_q[ALOADS], a_r[ALOADS], a_j[ALOADS];
#pragma unroll
  for (int i = 0; i < ALOADS; ++i) {
    const int idx = tid + i * 256;
    a_row[i] = idx >> 2; a_q[i] = idx & 3;
    const int m = m0 + a_row[i];
    a_r[i] = (m < M && a_row[i] < BM) ? m / a.Tj : -1;
    a_j[i] = (m < M) ? m % a.Tj : 0;
  }
  const int kchunks = (cin + GBK - 1) / GBK;
  for (int tap = 0; tap < a.ntaps; ++tap) {
    const float* __restrict__ wt = a.w[tap];
    for (int kc = 0; kc < kchunks; ++kc) {
      const int ci0 = kc * GBK;
#pragma unroll
      for (int i = 0; i < ALOADS; ++i) {
        if (a_row[i] < BM) {
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          const int c = ci0 + a_q[i] * 4;
          const int ti = a_j[i] * a.istride + a.ioff[tap];
          if (a_r[i] >= 0 && c < cin && ti >= 0 && ti < a.Tin) {
            const float* p = (c < a.c0) ? a.in0 + ((size_t)a_r[i] * a.Tin + ti) * a.c0 + c
                                        : a.in1 + ((size_t)a_r[i] * a.Tin + ti) * a.c1 + (c - a.c0);
            v = *reinterpret_cast<const float4*>(p);
          }
          As[a_q[i] * 4 + 0][a_row[i]] = v.x; As[a_q[i] * 4 + 1][a_row[i]] = v.y;
          As[a_q[i] * 4 + 2][a_row[i]] = v.z; As[a_q[i] * 4 + 3][a_row[i]] = v.w;
        }
      }
      if (!TRANSB) {
        const int b_k = tid >> 4, b_n = (tid & 15) * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        const int c = ci0 + b_k, n = n0 + b_n;
        if (c < cin && n < a.cout) v = *reinterpret_cast<const float4*>(wt + (size_t)c * a.ldw + n);
        *reinterpret_cast<float4*>(&Bs[b_k][b_n]) = v;
      } else {
        const int b_n = tid >> 2, b_k = (tid & 3) * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        const int c = ci0 + b_k, n = n0 + b_n;
        if (c < cin && n < a.cout) v = *reinterpret_cast<const float4*>(wt + (size_t)n * a.ldw + c);
        Bs[b_k + 0][b_n] = v.x; Bs[b_k + 1][b_n] = v.y; Bs[b_k + 2][b_n] = v.z; Bs[b_k + 3][b_n] = v.w;
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < GBK; ++k) {
        float av[RPT];
        if (RPT == 8) {
          const float4 a0 = *reinterpret_cast<const float4*>(&As[k][ty * 8]);
          const float4 a1 = *reinterpret_cast<const float4*>(&As[k][ty * 8 + 4]);
          av[0] = a0.x; av[1] = a0.y; av[2] = a0.z; av[3] = a0.w;
          av[RPT - 4] = a1.x; av[RPT - 3] = a1.y; av[RPT - 2] = a1.z; av[RPT - 1] = a1.w;
        } else if (RPT == 4) {
          const float4 a0 = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
          av[0] = a0.x; av[1] = a0.y; av[RPT - 2] = a0.z; av[RPT - 1] = a0.w;
        } else {
          const float2 a0 = *reinterpret_cast<const float2*>(&As[k][ty * 2]);
          av[0] = a0.x; av[RPT - 1] = a0.y;
        }
        const float4 b = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
        const float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int i = 0; i < RPT; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
      }
      __syncthreads();
    }
  }
  const int n = n0 + tx * 4;
  if (n < a.cout) {
    float4 bb = make_float4(0.f, 0.f, 0.f, 0.f);
    if (a.bias) bb = *reinterpret_cast<const float4*>(a.bias + n);
#pragma unroll
    for (int i = 0; i < RPT; ++i) {
      const int m = m0 + ty * RPT + i;
      if (m < M) {
        const int r = m / a.Tj, j = m % a.Tj;
        float4* op = reinterpret_cast<float4*>(a.out + ((size_t)r * a.Tout + j * a.ostride + a.ooff) * a.cout + n);
        float4 o = make_float4(acc[i][0] + bb.x, acc[i][1] + bb.y, acc[i][2] + bb.z, acc[i][3] + bb.w);
        if (a.accum) { const float4 p = *op; o.x += p.x; o.y += p.y; o.z += p.z; o.w += p.w; }
        *op = o;
      }
    }
  }
}

template <bool TRANSB>
static int tgemm_launch(CldHandle* h, const TGemm& a, int n_out, cudaStream_t s) {
  const int M = a.R * a.Tj, ny = (n_out + GBN - 1) / GBN;
  const int want = 2 * h->num_sms;
  if (((M + 127) / 128) * ny >= want) tgemm_kernel<TRANSB, 128><<<dim3((M + 127) / 128, ny), 256, 0, s>>>(a);
  else if (((M + 63) / 64) * ny >= want) tgemm_kernel<TRANSB, 64><<<dim3((M + 63) / 64, ny), 256, 0, s>>>(a);
  else tgemm_kernel<TRANSB, 32><<<dim3((M + 31) / 32, ny), 256, 0, s>>>(a);
  CLD_LAUNCH_OK(h, TRANSB ? "tgemm_kernel<dgrad>" : "tgemm_kernel<fwd>");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// weight gradient: dW[tap][ci][co] = sum_m in[m @ tap][ci] * dOut[m][co], M split over grid.z, partials reduced in fixed order
// ------------------------------------------------------------------------------------------------
struct TWgrad {
  const float* in0; int c0; const float* in1; int c1; int Tin;
  const float* dout; int Tout; int cout;
  int ntaps; int ioff[5]; int istride, ostride, ooff;
  int Tj; int R;
  float* part;                  // [splits][ntaps][cin][cout]
  float* bias_part;             // [splits][cout] column sums of dOut (the bias gradient), or nullptr
  int splits, chunk;            // chunk = rows of M per split (multiple of 16)
};

__global__ void __launch_bounds__(256) twgrad_kernel(TWgrad a) {
  __shared__ __align__(16) float As[16][64 + 4];
  __shared__ __align__(16) float Bs[16][64 + 4];
  const int tid = threadIdx.x;
  const int ci0 = blockIdx.x * 64, co0 = blockIdx.y * 64;
  const int tap = blockIdx.z % a.ntaps, split = blockIdx.z / a.ntaps;
  const int cin = a.c0 + a.c1;
  const int M = a.R * a.Tj;
  const int m_lo = split * a.chunk, m_hi = min(M, m_lo + a.chunk);
  const int ty = tid >> 4, tx = tid & 15;
  const int l_row = tid >> 4, l_c = (tid & 15) * 4;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  const bool do_bias = a.bias_part && blockIdx.x == 0 && tap == 0;     // one CTA per (output-channel tile, split) also sums dOut
  float4 bs = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int mb = m_lo; mb < m_hi; mb += 16) {
    const int m = mb + l_row;
    float4 va = make_float4(0.f, 0.f, 0.f, 0.f), vb = va;
    if (m < m_hi) {
      const int r = m / a.Tj, j = m - r * a.Tj;
      const int ti = j * a.istride + a.ioff[tap];
      const int c = ci0 + l_c;
      if (c < cin && ti >= 0 && ti < a.Tin) {
        const float* p = (c < a.c0) ? a.in0 + ((size_t)r * a.Tin + ti) * a.c0 + c
                                    : a.in1 + ((size_t)r * a.Tin + ti) * a.c1 + (c - a.c0);
        va = *reinterpret_cast<const float4*>(p);
      }
      const int n = co0 + l_c;
      if (n < a.cout) vb = *reinterpret_cast<const float4*>(a.dout + ((size_t)r * a.Tout + j * a.ostride + a.ooff) * a.cout + n);
    }
    *reinterpret_cast<float4*>(&As[l_row][l_c]) = va;
    *reinterpret_cast<float4*>(&Bs[l_row][l_c]) = vb;
    if (do_bias) { bs.x += vb.x; bs.y += vb.y; bs.z += vb.z; bs.w += vb.w; }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const float4 x = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 y = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float xv[4] = {x.x, x.y, x.z, x.w}, yv[4] = {y.x, y.y, y.z, y.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(xv[i], yv[j], acc[i][j]);
    }
    __syncthreads();
  }
  const int n = co0 + tx * 4;
  if (n < a.cout) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int ci = ci0 + ty * 4 + i;
      if (ci < cin)
        *reinterpret_cast<float4*>(a.part + (((size_t)split * a.ntaps + tap) * cin + ci) * a.cout + n) =
            make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
    }
  }
  if (do_bias) {                                       // 16 row-threads per column quad, summed in a fixed order
    *reinterpret_cast<float4*>(&Bs[l_row][l_c]) = bs;
    __syncthreads();
    if (tid < 64 && co0 + tid < a.cout) {
      float t = 0.f;
#pragma unroll
      for (int r = 0; r < 16; ++r) t += Bs[r][tid];
      a.bias_part[(size_t)split * a.cout + co0 + tid] = t;
    }
  }
}

// sum the split partials (fixed order) and write the gradient in the reference's parameter layout:
//   Conv1d / Linear  [cout][cin][K]   (transposed = 0)      ConvTranspose1d  [cin][cout][K]   (transposed = 1)
// The columns [co_off, co_off + co_n) of the packed matrix are written (a slice for the concatenated time-bias projection).
struct TKs { int k[5]; };
__global__ void __launch_bounds__(256) twreduce_kernel(const float* __restrict__ part, int splits, int ntaps, int cin, int cout,
                                                       int co_off, int co_n, float* __restrict__ dst, int K, TKs ks, int transposed,
                                                       const float* __restrict__ bias_part, float* __restrict__ bias_dst) {
  const int idx = blockIdx.x * 256 + threadIdx.x;
  const int total = ntaps * cin * co_n;
  if (idx >= total) {
    const int c = idx - total;
    if (bias_dst && c < co_n) {
      float s = 0.f;
      for (int i = 0; i < splits; ++i) s += bias_part[(size_t)i * cout + co_off + c];
      bias_dst[c] = s;
    }
    return;
  }
  const int co = idx % co_n, ci = (idx / co_n) % cin, tap = idx / (co_n * cin);
  const size_t stride = (size_t)ntaps * cin * cout;
  const float* p = part + ((size_t)tap * cin + ci) * cout + co_off + co;
  float s = 0.f;
  for (int i = 0; i < splits; ++i) s += p[i * stride];
  const int k = ks.k[tap];
  if (transposed) dst[((size_t)ci * co_n + co) * K + k] = s;
  else dst[((size_t)co * cin + ci) * K + k] = s;
}

// ------------------------------------------------------------------------------------------------
// column sums of a [M, C] matrix (bias / affine / time-bias gradients): two stages, fixed order
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ src, int M, int C, float* __restrict__ partial) {
  const int c = blockIdx.y * 256 + threadIdx.x;
  if (c >= C) return;
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  int m = blockIdx.x;
  const int st = gridDim.x;
  for (; m + 3 * st < M; m += 4 * st) {
    s0 += src[(size_t)m * C + c]; s1 += src[(size_t)(m + st) * C + c];
    s2 += src[(size_t)(m + 2 * st) * C + c]; s3 += src[(size_t)(m + 3 * st) * C + c];
  }
  for (; m < M; m += st) s0 += src[(size_t)m * C + c];
  partial[(size_t)blockIdx.x * C + c] = (s0 + s1) + (s2 + s3);
}
// columns [0, split) go to dst0, [split, 2 split) to dst1, [2 split, C) to dst2 (up to three gradient tensors from one pass); also
// used directly on a [M, C] matrix of few rows (nblk = M)
__global__ void __launch_bounds__(256) colsum_final_kernel(const float* __restrict__ partial, int nblk, int C, float* __restrict__ dst0,
                                                           int split, float* __restrict__ dst1, float* __restrict__ dst2) {
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c >= C) return;
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  int b = 0;
  for (; b + 3 < nblk; b += 4) {
    s0 += partial[(size_t)b * C + c]; s1 += partial[(size_t)(b + 1) * C + c];
    s2 += partial[(size_t)(b + 2) * C + c]; s3 += partial[(size_t)(b + 3) * C + c];
  }
  for (; b < nblk; ++b) s0 += partial[(size_t)b * C + c];
  const float s = (s0 + s1) + (s2 + s3);
  if (c < split) dst0[c] = s; else if (c < 2 * split) dst1[c - split] = s; else if (dst2) dst2[c - 2 * split] = s;
}

// few rows (the per-row partials of a minibatch): 32 columns x 8 row slices per CTA, slices added in a fixed order
__global__ void __launch_bounds__(256) colsum_small_kernel(const float* __restrict__ src, int M, int C, float* __restrict__ dst0, int split,
                                                           float* __restrict__ dst1, float* __restrict__ dst2) {
  __shared__ float red[8][32];
  const int cl = threadIdx.x & 31, part = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cl;
  float s = 0.f;
  if (c < C) {
    const int per = (M + 7) >> 3, lo = part * per, hi = min(M, lo + per);
    for (int m = lo; m < hi; ++m) s += src[(size_t)m * C + c];
  }
  red[part][cl] = s;
  __syncthreads();
  if (part == 0 && c < C) {
    float t = red[0][cl];
#pragma unroll
    for (int i = 1; i < 8; ++i) t += red[i][cl];
    if (c < split) dst0[c] = t; else if (c < 2 * split) dst1[c - split] = t; else if (dst2) dst2[c - 2 * split] = t;
  }
}

// ------------------------------------------------------------------------------------------------
// elementwise helpers
// ------------------------------------------------------------------------------------------------
// dst[m, c] (+)= src[m * ld + off + c]
__global__ void __launch_bounds__(256) slice_kernel(float* __restrict__ dst, const float* __restrict__ src, size_t n, int C, int ld,
                                                    int off, int add) {
  const size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  const size_t m = i / C;
  const int c = (int)(i - m * C);
  const float v = src[m * ld + off + c];
  dst[i] = add ? dst[i] + v : v;
}

__device__ __forceinline__ float softplus_f(float x) { return (x > 20.f) ? x : log1pf(expf(x)); }
__device__ __forceinline__ float mish_fwd(float x) { return x * tanhf(softplus_f(x)); }
// d/dx [x tanh(softplus(x))] = tanh(sp) + x sigmoid(x) (1 - tanh(sp)^2)   (ATen mish_backward)
__device__ __forceinline__ float mish_grad(float x) {
  const float tsp = tanhf(softplus_f(x));
  const float sig = 1.f / (1.f + expf(-x));
  return fmaf(x * sig, 1.f - tsp * tsp, tsp);
}

// ------------------------------------------------------------------------------------------------
// backward of GroupNorm(8) -> Mish -> (+ time bias | + residual)        (diffuser_helpers.py:58-64, temporal.py:37-45)
//   x = conv output [R,T,C];  xh = (x - mean) rstd;  u = xh g + b;  y = mish(u) (+ ...)
//   dU = dY mish'(u);  dg[c] += dU xh;  db[c] += dU;  dxh = dU g;  dx = rstd (dxh - mean(dxh) - xh mean(dxh xh))
// One CTA per row, warp = group.  cpg divides 32, so a lane always meets the same channel: per-channel sums stay in registers.
// Per-row partials (rp [R][dg | db | sum_t dx = the bias gradient of the convolution in front], and sum_t dY = d(time bias)) are
// written; one colsum reduces them over the rows.
// ------------------------------------------------------------------------------------------------
// NW warps share a group (a 128-row minibatch is one CTA per row on 128 of 148 SMs: the per-warp loop of 13..26 dependent
// load -> libm-Mish iterations is the kernel's latency; more warps per group shorten it).  Partial sums of the NW warps are combined
// through shared memory in a fixed order.
template <int NW>
__device__ __forceinline__ float group_sum(float v, float* red, int g, int w, int lane) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if (lane == 0) red[g * NW + w] = v;
  __syncthreads();
  float t = red[g * NW];
#pragma unroll
  for (int i = 1; i < NW; ++i) t += red[g * NW + i];
  return t;
}

// forward: GroupNorm(8) -> Mish -> (+ per-row channel bias | + residual), as gn_mish_fp32 (kernels_unet_fp32.cu) with NW warps per group
template <int NW>
__global__ void __launch_bounds__(256 * NW) gn_mish_fwd_mw_kernel(const float* __restrict__ in, const float* __restrict__ gamma,
                                                                   const float* __restrict__ beta, const float* __restrict__ tbias,
                                                                   int tb_stride, const float* __restrict__ res, float* __restrict__ out,
                                                                   int T, int C) {
  __shared__ float red[2][8 * NW];
  const int r = blockIdx.x, wid = threadIdx.x >> 5, g = wid / NW, w = wid % NW, lane = threadIdx.x & 31;
  const int cpg = C >> 3, n = T * cpg;
  const float* xin = in + (size_t)r * T * C + g * cpg;
  float s = 0.f;
  for (int e = lane + 32 * w; e < n; e += 32 * NW) s += xin[(e / cpg) * C + (e % cpg)];
  const float mean = group_sum<NW>(s, red[0], g, w, lane) / (float)n;
  float v = 0.f;
  for (int e = lane + 32 * w; e < n; e += 32 * NW) {
    const float d = xin[(e / cpg) * C + (e % cpg)] - mean;
    v = fmaf(d, d, v);
  }
  const float rstd = 1.0f / sqrtf(group_sum<NW>(v, red[1], g, w, lane) / (float)n + 1e-5f);
  for (int e = lane + 32 * w; e < n; e += 32 * NW) {
    const int t = e / cpg, c = g * cpg + (e % cpg);
    float y = (xin[t * C + (e % cpg)] - mean) * rstd * gamma[c] + beta[c];
    y = mish_fwd(y);
    if (tbias) y += tbias[(size_t)r * tb_stride + c];
    if (res) y += res[((size_t)r * T + t) * C + c];
    out[((size_t)r * T + t) * C + c] = y;
  }
}

template <int NW>
__global__ void __launch_bounds__(256 * NW) gn_mish_bwd_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                                                const float* __restrict__ beta, const float* __restrict__ dy,
                                                                float* __restrict__ dx, float* __restrict__ rp,
                                                                float* __restrict__ dtb, int tb_stride, int T, int C) {
  __shared__ float red[4][8 * NW];
  __shared__ float chan[4][8 * NW][32];             // per-warp per-channel partials of dgamma, dbeta, sum dY, sum dx
  const int r = blockIdx.x, wid = threadIdx.x >> 5, g = wid / NW, w = wid % NW, lane = threadIdx.x & 31;
  const int cpg = C >> 3, n = T * cpg;
  const size_t base = (size_t)r * T * C + g * cpg;
  const float* xin = x + base;
  const float* dyin = dy + base;
  float* dxo = dx + base;
  const int e0 = lane + 32 * w, es = 32 * NW;
  float s = 0.f;
  for (int e = e0; e < n; e += es) s += xin[(e / cpg) * C + (e % cpg)];
  const float mean = group_sum<NW>(s, red[0], g, w, lane) / (float)n;
  float v = 0.f;
  for (int e = e0; e < n; e += es) {
    const float d = xin[(e / cpg) * C + (e % cpg)] - mean;
    v = fmaf(d, d, v);
  }
  const float rstd = 1.0f / sqrtf(group_sum<NW>(v, red[1], g, w, lane) / (float)n + 1e-5f);
  const int cl = lane % cpg, c = g * cpg + cl;        // this lane's channel (cpg | 32, and the warp stride 32 NW keeps it)
  const float gm = gamma[c], bt = beta[c];
  float sg = 0.f, sb = 0.f, sy = 0.f, s1 = 0.f, s2 = 0.f;
  for (int e = e0; e < n; e += es) {
    const int off = (e / cpg) * C + cl;
    const float xh = (xin[off] - mean) * rstd;
    const float u = fmaf(xh, gm, bt);
    const float gy = dyin[off];
    const float du = gy * mish_grad(u);
    const float dxh = du * gm;
    sg = fmaf(du, xh, sg); sb += du; sy += gy;
    s1 += dxh; s2 = fmaf(dxh, xh, s2);
    dxo[off] = dxh;
  }
  // per-channel sums: lanes with equal lane % cpg, then the NW warps of the group
  for (int o = 16; o >= cpg; o >>= 1) {
    sg += __shfl_xor_sync(0xffffffffu, sg, o); sb += __shfl_xor_sync(0xffffffffu, sb, o); sy += __shfl_xor_sync(0xffffffffu, sy, o);
  }
  if (lane < cpg) { chan[0][wid][lane] = sg; chan[1][wid][lane] = sb; chan[2][wid][lane] = sy; }
  const float m1 = group_sum<NW>(s1, red[2], g, w, lane) / (float)n;        // (its __syncthreads also publishes chan[0..2])
  const float m2 = group_sum<NW>(s2, red[3], g, w, lane) / (float)n;
  if (w == 0 && lane < cpg) {
    float tg = 0.f, tb = 0.f, ty = 0.f;
#pragma unroll
    for (int i = 0; i < NW; ++i) { tg += chan[0][g * NW + i][lane]; tb += chan[1][g * NW + i][lane]; ty += chan[2][g * NW + i][lane]; }
    rp[(size_t)r * 3 * C + c] = tg; rp[(size_t)r * 3 * C + C + c] = tb;      // [R][gamma | beta | conv bias]
    if (dtb) dtb[(size_t)r * tb_stride + c] = ty;
  }
  float sx = 0.f;                                     // sum_t dx of this lane's channel = the row's share of the conv bias gradient
  for (int e = e0; e < n; e += es) {
    const int off = (e / cpg) * C + cl;
    const float xh = (xin[off] - mean) * rstd;
    const float d = rstd * (dxo[off] - m1 - xh * m2);
    dxo[off] = d;
    sx += d;
  }
  for (int o = 16; o >= cpg; o >>= 1) sx += __shfl_xor_sync(0xffffffffu, sx, o);
  if (lane < cpg) chan[3][wid][lane] = sx;
  __syncthreads();
  if (w == 0 && lane < cpg) {
    float tx = 0.f;
#pragma unroll
    for (int i = 0; i < NW; ++i) tx += chan[3][g * NW + i][lane];
    rp[(size_t)r * 3 * C + 2 * C + c] = tx;
  }
}

// ------------------------------------------------------------------------------------------------
// backward of the time MLP (temporal.py:74-79): emb -> Linear(d,4d) -> Mish -> Linear(4d,d), then the block-side Mish.
// dtm [R, ld] holds d(loss)/d(Mish(time embedding)) in its first d columns.  Writes the operands of the two weight-gradient GEMMs.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) time_mlp_bwd_kernel(const int64_t* __restrict__ t, const float* __restrict__ w1,
                                                           const float* __restrict__ b1, const float* __restrict__ w2,
                                                           const float* __restrict__ b2, const float* __restrict__ freqs,
                                                           const float* __restrict__ dtm, int ld, float* __restrict__ emb_o,
                                                           float* __restrict__ hid_o, float* __restrict__ dpre1_o,
                                                           float* __restrict__ dpre2_o, int d) {
  __shared__ float emb[64], pre1[256], hid[256], dp2[64];
  const int r = blockIdx.x, tid = threadIdx.x;
  const float tv = (float)t[r];
  const int half = d >> 1;
  if (tid < d) {
    const float a = tv * freqs[tid % half];
    emb[tid] = (tid < half) ? sinf(a) : cosf(a);
    emb_o[(size_t)r * d + tid] = emb[tid];
  }
  __syncthreads();
  for (int o = tid; o < 4 * d; o += blockDim.x) {
    float acc = b1[o];
    for (int k = 0; k < d; ++k) acc = fmaf(w1[o * d + k], emb[k], acc);
    pre1[o] = acc; hid[o] = mish_fwd(acc);
    hid_o[(size_t)r * 4 * d + o] = hid[o];
  }
  __syncthreads();
  if (tid < d) {
    float acc = b2[tid];
    for (int k = 0; k < 4 * d; ++k) acc = fmaf(w2[tid * 4 * d + k], hid[k], acc);
    const float g = dtm[(size_t)r * ld + tid] * mish_grad(acc);
    dp2[tid] = g;
    dpre2_o[(size_t)r * d + tid] = g;
  }
  __syncthreads();
  for (int o = tid; o < 4 * d; o += blockDim.x) {
    float acc = 0.f;
    for (int k = 0; k < d; ++k) acc = fmaf(w2[k * 4 * d + o], dp2[k], acc);
    dpre1_o[(size_t)r * 4 * d + o] = acc * mish_grad(pre1[o]);
  }
}

// ------------------------------------------------------------------------------------------------
// loss heads
// ------------------------------------------------------------------------------------------------
// PPO clipped surrogate on log_prob (guide_dm_trainer.py:150-168 with dm_model.py:165-174), one CTA per row:
//   mean = c1[t] x_t - c2[t] eps;  logp = mean_{T,D} Normal(mean, sigma[t]).log_prob(x_tm1);  ratio = exp(logp - logp_old)
//   loss = -(1/R) sum_r min(ratio A, clamp(ratio, 1-e, 1+e) A),  A = reward - baseline
// d_eps = dloss/deps (torch.min sends the gradient to the smaller argument; inside the clip range both arguments carry it).
__global__ void __launch_bounds__(128) ppo_head_kernel(const float* __restrict__ eps, const float* __restrict__ x_t,
                                                       const float* __restrict__ x_tm1, const int64_t* __restrict__ t,
                                                       const float* __restrict__ sched, int n_t, const float* __restrict__ logp_old,
                                                       const float* __restrict__ reward, float baseline,
                                                       const float* __restrict__ baseline_dev, float clip,
                                                       float* __restrict__ logp_new, float* __restrict__ loss_row,
                                                       float* __restrict__ d_eps, int n, int R) {
  __shared__ float red[4];
  const int r = blockIdx.x, tid = threadIdx.x;
  int tt = (int)t[r];
  tt = tt < 0 ? 0 : (tt >= n_t ? n_t - 1 : tt);
  const float c1 = sched[tt], c2 = sched[n_t + tt], lv = sched[2 * n_t + tt];
  const float sigma = expf(0.5f * lv), var = sigma * sigma;
  const size_t base = (size_t)r * n;
  float s = 0.f;
  for (int i = tid; i < n; i += 128) {
    const float mean = c1 * x_t[base + i] - c2 * eps[base + i];
    const float d = x_tm1[base + i] - mean;
    s += -(d * d) / (2.f * var) - logf(sigma) - 0.91893853320467274f;
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((tid & 31) == 0) red[tid >> 5] = s;
  __syncthreads();
  const float logp = ((red[0] + red[1]) + (red[2] + red[3])) / (float)n;
  const float ratio = expf(logp - logp_old[r]);
  const float A = reward[r] - (baseline_dev ? baseline_dev[0] : baseline);
  const float s1 = ratio * A, s2 = fminf(fmaxf(ratio, 1.f - clip), 1.f + clip) * A;
  const bool inside = ratio >= 1.f - clip && ratio <= 1.f + clip;
  float gl = 0.f;                                   // d min(s1, s2) / d logp
  if (inside || s1 < s2) gl = s1;
  else if (s1 == s2) gl = 0.5f * s1;
  if (tid == 0) {
    if (logp_new) logp_new[r] = logp;
    loss_row[r] = -fminf(s1, s2) / (float)R;
  }
  if (d_eps) {
    const float k = (-gl / (float)R) * (-c2) / (var * (float)n);
    for (int i = tid; i < n; i += 128) {
      const float mean = c1 * x_t[base + i] - c2 * eps[base + i];
      d_eps[base + i] = k * (x_tm1[base + i] - mean);
    }
  }
}

// F.mse_loss(noise, eps) of DmModel.compute_losses (dm_model.py:83-90): loss_row[r] = sum_i (eps - noise)^2 / (R n)
__global__ void __launch_bounds__(128) mse_head_kernel(const float* __restrict__ eps, const float* __restrict__ noise,
                                                       float* __restrict__ loss_row, float* __restrict__ d_eps, int n, int R) {
  __shared__ float red[4];
  const int r = blockIdx.x, tid = threadIdx.x;
  const size_t base = (size_t)r * n;
  const float inv = 1.f / ((float)R * (float)n);
  float s = 0.f;
  for (int i = tid; i < n; i += 128) {
    const float d = eps[base + i] - noise[base + i];
    s = fmaf(d, d, s);
    if (d_eps) d_eps[base + i] = 2.f * d * inv;
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((tid & 31) == 0) red[tid >> 5] = s;
  __syncthreads();
  if (tid == 0) loss_row[r] = ((red[0] + red[1]) + (red[2] + red[3])) * inv;
}

// one CTA: out[0] = sum_r v[r] (fixed order)
__global__ void __launch_bounds__(256) sum_rows_kernel(const float* __restrict__ v, int R, float* __restrict__ out) {
  __shared__ float red[256];
  float s = 0.f;
  for (int i = threadIdx.x; i < R; i += 256) s += v[i];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = red[0];
}

// torch.optim.Adam (no amsgrad; weight_decay added to the gradient), one flat parameter vector
__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                   float* __restrict__ v, size_t n, float step_size, float w1, float b2, float w2, float eps,
                                                   float wd, float bc2_sqrt, const float* __restrict__ dyn) {
  const size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  if (dyn) { step_size = dyn[0]; bc2_sqrt = dyn[1]; }
  const float pi = p[i];
  const float gi = fmaf(wd, pi, g[i]);
  const float mi = m[i] + (gi - m[i]) * w1;                       // torch: exp_avg.lerp_(grad, 1 - beta1)
  const float vi = fmaf(b2, v[i], w2 * gi * gi);                  // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
  m[i] = mi; v[i] = vi;
  const float denom = sqrtf(vi) / bc2_sqrt + eps;
  p[i] = pi - step_size * (mi / denom);
}

// step counter and learning rate live on the device (a CUDA graph of the update replays with changing step / lr): one thread
// advances the step and derives the two scalars of this step in double, as torch does on the host
__global__ void adam_tick_kernel(long long* __restrict__ step, const double* __restrict__ lr, double b1, double b2, float* __restrict__ dyn) {
  const long long st = ++step[0];
  dyn[0] = (float)(lr[0] / (1.0 - pow(b1, (double)st)));
  dyn[1] = (float)sqrt(1.0 - pow(b2, (double)st));
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
struct BlkStash { const float* in0; int c0; const float* in1; int c1; int T; float *A0, *B0, *A1, *OUT; };

struct TrainState {
  int cap_rows = 0;
  float* arena = nullptr;
  BlkStash blk[12];
  float *p0 = nullptr, *p1 = nullptr, *q0 = nullptr, *q1 = nullptr, *fA = nullptr, *fB = nullptr, *tmpR = nullptr;
  float *gB = nullptr, *gcat8 = nullptr, *gcat10 = nullptr;
  // The parameter gradients (weight-gradient GEMMs, split reductions, column sums) run on a second stream beside the data-gradient
  // chain.  What they read is never overwritten during a backward: every GroupNorm backward has its own dA / per-row partial buffers,
  // every layer its own data-gradient buffer; the scratch they share (part, bias_part, colpart) is touched by that stream only.
  static constexpr int MAX_UNITS = 26, MAX_GD = 20, N_EVENTS = 64;
  float* gA_u[MAX_UNITS] = {nullptr};
  float* rp_u[MAX_UNITS] = {nullptr};
  float* gD[MAX_GD] = {nullptr};
  int unit = 0, nd = 0;
  cudaStream_t aux = nullptr;
  cudaEvent_t evs[N_EVENTS] = {nullptr};
  unsigned ev_next = 0;
  float *dtbias = nullptr, *dtcm = nullptr, *emb = nullptr, *hid = nullptr, *dpre1 = nullptr, *dpre2 = nullptr;
  float *loss_row = nullptr, *deps = nullptr;
  float* part = nullptr;  size_t part_floats = 0;
  float* colpart = nullptr;
  float* bias_part = nullptr;      // [MAX_SPLITS][256] split partials of a convolution's bias gradient
  float* tb_bgrad = nullptr;       // [tb_total] bias gradient of the concatenated time / cond projection
  float* sched_dev = nullptr;
  unsigned long long sched_version = ~0ull;     // h->sched_version the device copy was made from
  float* adam_dyn = nullptr;                    // [2] step size, sqrt of the second bias correction (graph-replayable Adam)
  const float* x = nullptr;
  const int64_t* t = nullptr;
  int R = 0;
  bool fwd_valid = false;
};

static TrainState* ts_of(CldHandle* h) { return reinterpret_cast<TrainState*>(h->train); }

void train_destroy(CldHandle* h) {
  TrainState* st = ts_of(h);
  if (!st) return;
  if (st->arena) cudaFree(st->arena);
  if (st->part) cudaFree(st->part);
  if (st->colpart) cudaFree(st->colpart);
  if (st->bias_part) cudaFree(st->bias_part);
  if (st->sched_dev) cudaFree(st->sched_dev);
  if (st->adam_dyn) cudaFree(st->adam_dyn);
  if (st->aux) cudaStreamDestroy(st->aux);
  for (cudaEvent_t e : st->evs)
    if (e) cudaEventDestroy(e);
  delete st;
  h->train = nullptr;
}

void train_invalidate(CldHandle* h) {
  if (TrainState* st = ts_of(h)) st->fwd_valid = false;
}

constexpr int COLSUM_BLOCKS = 128;
constexpr int MAX_SPLITS = 1024;
constexpr size_t PART_FLOATS = (size_t)6 << 20;

static int train_prepare(CldHandle* h, int R) {
  if (!h->train) h->train = new TrainState();
  TrainState* st = ts_of(h);
  const CldConfig& c = h->cfg;
  const int tb_total = h->unet.tb_total;
  if (!st->part) {
    CLD_CUDA_OK(h, cudaMalloc((void**)&st->part, PART_FLOATS * sizeof(float)));
    st->part_floats = PART_FLOATS;
    CLD_CUDA_OK(h, cudaMalloc((void**)&st->colpart, (size_t)(COLSUM_BLOCKS + 1) * CLD_TB_TOTAL_MAX * sizeof(float)));
    st->tb_bgrad = st->colpart + (size_t)COLSUM_BLOCKS * CLD_TB_TOTAL_MAX;
    CLD_CUDA_OK(h, cudaMalloc((void**)&st->bias_part, (size_t)MAX_SPLITS * 256 * sizeof(float)));
    if (!h->env_train_serial) {
      CLD_CUDA_OK(h, cudaStreamCreateWithFlags(&st->aux, cudaStreamNonBlocking));
      for (cudaEvent_t& e : st->evs) CLD_CUDA_OK(h, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    CLD_CUDA_OK(h, cudaMalloc((void**)&st->sched_dev, (size_t)3 * c.n_timesteps * sizeof(float)));
    CLD_CUDA_OK(h, cudaMalloc((void**)&st->adam_dyn, 2 * sizeof(float)));
  }
  if (R <= st->cap_rows) return 0;
  if (st->arena) { cudaFree(st->arena); st->arena = nullptr; st->cap_rows = 0; }
  const size_t E = h->act_elems;                 // per-row elements of the largest activation
  const int td = c.base_dim;
  for (int i = 0; i < 3; ++i) {
    const int cpg = c.dims[i] / 8;
    if (c.dims[i] > 256 || (cpg != 1 && cpg != 2 && cpg != 4 && cpg != 8 && cpg != 16 && cpg != 32))
      return fail(h, CLD_ERR_UNSUPPORTED, "the denoiser backward needs dims of 8 x {1,2,4,8,16,32} channels");
  }
  if (tb_total > CLD_TB_TOTAL_MAX) return fail(h, CLD_ERR_UNSUPPORTED, "time-bias width %d above %d", tb_total, CLD_TB_TOTAL_MAX);
  if (td > 64) return fail(h, CLD_ERR_UNSUPPORTED, "the denoiser backward needs base_dim <= 64");
  // 12 blocks x 4 + p0 p1 q0 q1 fA fB tmpR + gB + 2 x 2 (concat gradients) = 60 E, + 26 dA + 20 data-gradient buffers, + the small per-row vectors
  const size_t per_row = (60 + TrainState::MAX_UNITS + TrainState::MAX_GD) * E + (size_t)TrainState::MAX_UNITS * 768 + (size_t)tb_total + 64 + td + 4 * td + 4 * td + td + 1 + (size_t)c.horizon * c.latent_dim;
  const size_t cap = (size_t)R;
  CLD_CUDA_OK(h, cudaMalloc((void**)&st->arena, per_row * cap * sizeof(float)));
  float* p = st->arena;
  auto take = [&](size_t per) { float* q = p; p += per * cap; return q; };
  for (int b = 0; b < 12; ++b) { st->blk[b].A0 = take(E); st->blk[b].B0 = take(E); st->blk[b].A1 = take(E); st->blk[b].OUT = take(E); }
  st->p0 = take(E); st->p1 = take(E); st->q0 = take(E); st->q1 = take(E); st->fA = take(E); st->fB = take(E); st->tmpR = take(E);
  st->gB = take(E); st->gcat8 = take(2 * E); st->gcat10 = take(2 * E);
  for (int i = 0; i < TrainState::MAX_UNITS; ++i) { st->gA_u[i] = take(E); st->rp_u[i] = take(768); }
  for (int i = 0; i < TrainState::MAX_GD; ++i) st->gD[i] = take(E);
  st->dtbias = take(tb_total); st->dtcm = take(64); st->emb = take(td); st->hid = take(4 * td); st->dpre1 = take(4 * td);
  st->dpre2 = take(td); st->loss_row = take(1);
  st->deps = take((size_t)c.horizon * c.latent_dim);
  st->cap_rows = R;
  st->fwd_valid = false;
  return 0;
}

static const int kOff5[5] = {-2, -1, 0, 1, 2};
static const int kOff3[5] = {-1, 0, 1, 0, 0};
static const int kOff1[5] = {0, 0, 0, 0, 0};

// the parameter-gradient stream, ordered after everything enqueued on `s` so far (or `s` itself under CLD_TRAIN_SERIAL=1)
static cudaStream_t pg_stream(CldHandle* h, cudaStream_t s) {
  TrainState* st = ts_of(h);
  if (!st->aux) return s;
  cudaEvent_t e = st->evs[st->ev_next++ % TrainState::N_EVENTS];
  cudaEventRecord(e, s);
  cudaStreamWaitEvent(st->aux, e, 0);
  return st->aux;
}
// the caller's stream waits for the parameter-gradient stream
static void pg_join(CldHandle* h, cudaStream_t s) {
  TrainState* st = ts_of(h);
  if (!st->aux) return;
  cudaEvent_t e = st->evs[st->ev_next++ % TrainState::N_EVENTS];
  cudaEventRecord(e, st->aux);
  cudaStreamWaitEvent(s, e, 0);
}

// forward convolution  out = conv(in) (+ bias)
static int conv_fwd(CldHandle* h, const ConvW& w, const float* in0, int c0, const float* in1, int c1, int Tin, float* out, int Tout,
                    int Tj, int istride, int ostride, int ooff, const int* ioff, const float* bias, int R, cudaStream_t s) {
  if (h->train_tf32 && w.wt && tfconv_supported(c0, c1, w.cout, Tj)) {
    const int taps[5] = {0, 1, 2, 3, 4};
    return tfconv_launch(h, in0, c0, in1, c1, Tin, istride, Tj, w.wt, w.ntaps, w.ntaps, taps, ioff, bias, out, Tout, ostride, ooff, w.cout, 0, R, s);
  }
  TGemm a;
  a.in0 = in0; a.c0 = c0; a.in1 = in1; a.c1 = c1; a.Tin = Tin;
  for (int i = 0; i < 5; ++i) { a.w[i] = w.w + (size_t)(i < w.ntaps ? i : 0) * w.cin * w.cout; a.ioff[i] = i < w.ntaps ? ioff[i] : 0; }
  a.ldw = w.cout; a.bias = bias; a.out = out; a.Tout = Tout; a.cout = w.cout; a.ntaps = w.ntaps;
  a.istride = istride; a.ostride = ostride; a.ooff = ooff; a.Tj = Tj; a.R = R; a.accum = 0;
  return tgemm_launch<false>(h, a, w.cout, s);
}

// data gradient: out[r, j*ostride+ooff, 0:n_out) (+)= sum_i dout[r, j*istride+ioff[i], :] @ W[taps[i]]^T
static int conv_dgrad(CldHandle* h, const ConvW& w, int ntaps, const int* taps, const int* ioff, const float* dout, int Tdout,
                      float* out, int Tout, int n_out, int Tj, int istride, int ostride, int ooff, int accum, int R, cudaStream_t s) {
  if (h->train_tf32 && (n_out == w.cin || w.ntaps == 1) && tfconv_supported(w.cout, 0, n_out, Tj))
    return tfconv_launch(h, dout, w.cout, nullptr, 0, Tdout, istride, Tj, w.w, w.ntaps, ntaps, taps, ioff, nullptr, out, Tout, ostride, ooff,
                         n_out, accum, R, s);
  TGemm a;
  a.in0 = dout; a.c0 = w.cout; a.in1 = nullptr; a.c1 = 0; a.Tin = Tdout;
  for (int i = 0; i < 5; ++i) { a.w[i] = w.w + (size_t)taps[i < ntaps ? i : 0] * w.cin * w.cout; a.ioff[i] = i < ntaps ? ioff[i] : 0; }
  a.ldw = w.cout; a.bias = nullptr; a.out = out; a.Tout = Tout; a.cout = n_out; a.ntaps = ntaps;
  a.istride = istride; a.ostride = ostride; a.ooff = ooff; a.Tj = Tj; a.R = R; a.accum = accum;
  return tgemm_launch<true>(h, a, n_out, s);
}

// weight gradient of one packed matrix [ntaps][cin][cout] -> partials in st->part; `splits_out` for the reduce
static int conv_wgrad(CldHandle* h, int cin_total, int cout, int ntaps, const int* ioff, const float* in0, int c0, const float* in1,
                      int c1, int Tin, const float* dout, int Tdout, int Tj, int istride, int ostride, int ooff, int R,
                      int* splits_out, cudaStream_t s, bool with_bias = false, bool* bias_in_part = nullptr) {
  TrainState* st = ts_of(h);
  if (bias_in_part) *bias_in_part = false;
  if (h->train_tf32 && tfwgrad_supported(c0, c1, cout, Tj, R))        // tensor pipe; the caller sums dOut's columns itself
    return tfwgrad_launch(h, in0, c0, in1, c1, Tin, istride, Tj, dout, Tdout, ostride, ooff, cout, ntaps, ioff, st->part, st->part_floats,
                          MAX_SPLITS, R, splits_out, s);
  if (bias_in_part) *bias_in_part = with_bias;
  TWgrad a;
  a.in0 = in0; a.c0 = c0; a.in1 = in1; a.c1 = c1; a.Tin = Tin; a.dout = dout; a.Tout = Tdout; a.cout = cout; a.ntaps = ntaps;
  for (int i = 0; i < 5; ++i) a.ioff[i] = i < ntaps ? ioff[i] : 0;
  a.istride = istride; a.ostride = ostride; a.ooff = ooff; a.Tj = Tj; a.R = R; a.part = st->part;
  const int M = R * Tj;
  const int tiles = ((cin_total + 63) / 64) * ((cout + 63) / 64) * ntaps;
  int splits = (4 * h->num_sms + tiles - 1) / tiles;
  const int max_by_m = (M + 255) / 256;
  if (splits > max_by_m) splits = max_by_m;
  const size_t wsz = (size_t)ntaps * cin_total * cout;
  if ((size_t)splits * wsz > st->part_floats) splits = (int)(st->part_floats / wsz);
  if (splits > MAX_SPLITS) splits = MAX_SPLITS;
  if (splits < 1) return fail(h, CLD_ERR_UNSUPPORTED, "weight-gradient scratch too small");
  if (with_bias && cout > 256) return fail(h, CLD_ERR_UNSUPPORTED, "fused bias gradient needs cout <= 256");
  a.bias_part = with_bias ? st->bias_part : nullptr;
  int chunk = (M + splits - 1) / splits;
  chunk = (chunk + 15) / 16 * 16;
  splits = (M + chunk - 1) / chunk;
  a.splits = splits; a.chunk = chunk;
  dim3 grid((cin_total + 63) / 64, (cout + 63) / 64, ntaps * splits);
  twgrad_kernel<<<grid, 256, 0, s>>>(a);
  CLD_LAUNCH_OK(h, "twgrad_kernel");
  *splits_out = splits;
  return 0;
}

static int wreduce(CldHandle* h, int splits, int ntaps, int cin, int cout, int co_off, int co_n, float* dst, int K, const int* ks,
                   int transposed, cudaStream_t s, float* bias_dst = nullptr) {
  TKs k;
  for (int i = 0; i < 5; ++i) k.k[i] = i < ntaps ? ks[i] : 0;
  const int total = ntaps * cin * co_n + (bias_dst ? co_n : 0);
  twreduce_kernel<<<(total + 255) / 256, 256, 0, s>>>(ts_of(h)->part, splits, ntaps, cin, cout, co_off, co_n, dst, K, k, transposed,
                                                      ts_of(h)->bias_part, bias_dst);
  CLD_LAUNCH_OK(h, "twreduce_kernel");
  return 0;
}

static int colsum(CldHandle* h, const float* src, int M, int C, float* dst, cudaStream_t s, int split = -1, float* dst1 = nullptr,
                  float* dst2 = nullptr) {
  TrainState* st = ts_of(h);
  if (M <= 512) {                       // few rows (per-row partials of a minibatch): one pass
    colsum_small_kernel<<<(C + 31) / 32, 256, 0, s>>>(src, M, C, dst, split < 0 ? C : split, dst1, dst2);
    CLD_LAUNCH_OK(h, "colsum_small_kernel");
    return 0;
  }
  int nblk = (M + 31) / 32;
  if (nblk > COLSUM_BLOCKS) nblk = COLSUM_BLOCKS;
  dim3 grid(nblk, (C + 255) / 256);
  colsum_kernel<<<grid, 256, 0, s>>>(src, M, C, st->colpart);
  CLD_LAUNCH_OK(h, "colsum_kernel");
  colsum_final_kernel<<<(C + 255) / 256, 256, 0, s>>>(st->colpart, nblk, C, dst, split < 0 ? C : split, dst1, dst2);
  CLD_LAUNCH_OK(h, "colsum_final_kernel");
  return 0;
}

static int slice(CldHandle* h, float* dst, const float* src, size_t M, int C, int ld, int off, int add, cudaStream_t s) {
  const size_t n = M * C;
  slice_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(dst, src, n, C, ld, off, add);
  CLD_LAUNCH_OK(h, "slice_kernel");
  return 0;
}

// warps per GroupNorm group in the training kernels: 2 while the batch leaves SMs idle (latency), 1 for large batches (occupancy)
static int gn_mish_train(CldHandle* h, const float* in, const GnW& n, const float* tbias, int tb_stride, const float* res, float* out, int T,
                          int C, int R, cudaStream_t s) {
  if (R <= 2 * h->num_sms) gn_mish_fwd_mw_kernel<2><<<R, 512, 0, s>>>(in, n.g, n.b, tbias, tb_stride, res, out, T, C);
  else gn_mish_fwd_mw_kernel<1><<<R, 256, 0, s>>>(in, n.g, n.b, tbias, tb_stride, res, out, T, C);
  CLD_LAUNCH_OK(h, "gn_mish_fwd_mw_kernel");
  return 0;
}

static int block_fwd(CldHandle* h, int bi, const float* in0, int c0, const float* in1, int c1, int T, int R, cudaStream_t s) {
  TrainState* st = ts_of(h);
  const ResBlockW& rb = h->unet.rb[bi];
  BlkStash& b = st->blk[bi];
  b.in0 = in0; b.c0 = c0; b.in1 = in1; b.c1 = c1; b.T = T;
  int rc;
  if ((rc = conv_fwd(h, rb.c0, in0, c0, in1, c1, T, b.A0, T, T, 1, 1, 0, kOff5, rb.c0.b, R, s))) return rc;
  if ((rc = gn_mish_train(h, b.A0, rb.n0, h->tbias + rb.tb_off, h->unet.tb_total, nullptr, b.B0, T, rb.cout, R, s))) return rc;
  if ((rc = conv_fwd(h, rb.c1, b.B0, rb.cout, nullptr, 0, T, b.A1, T, T, 1, 1, 0, kOff5, rb.c1.b, R, s))) return rc;
  const float* res = in0;
  if (rb.res.w) {
    if ((rc = conv_fwd(h, rb.res, in0, c0, in1, c1, T, st->tmpR, T, T, 1, 1, 0, kOff1, rb.res.b, R, s))) return rc;
    res = st->tmpR;
  }
  return gn_mish_train(h, b.A1, rb.n1, nullptr, 0, res, b.OUT, T, rb.cout, R, s);
}

int unet_train_forward(CldHandle* h, const float* x, const float* cond, const int64_t* t, float* eps, int R, cudaStream_t s) {
  int rc;
  if ((rc = train_prepare(h, R))) return rc;
  TrainState* st = ts_of(h);
  const UnetW& u = h->unet;
  const CldConfig& c = h->cfg;
  const int T = c.horizon, T2 = T / 2, T4 = T / 4;
  const int d0 = c.dims[0], d1 = c.dims[1], d2 = c.dims[2], D = c.latent_dim;
  st->fwd_valid = false;
  // -> h->tcm, h->tbias (kept for the backward); the projection of all 12 blocks is one GEMM [R, 288] x [288, 1 792]
  const int tdim = c.base_dim + c.cond_dim;
  if (h->train_tf32 && u.tb_wt && tfconv_supported(tdim, 0, u.tb_total, 1)) {
    if ((rc = unet_time_cond(h, cond, t, R, s))) return rc;
    const int tap0[5] = {0, 0, 0, 0, 0};
    if ((rc = tfconv_launch(h, h->tcm, tdim, nullptr, 0, 1, 1, 1, u.tb_wt, 1, 1, tap0, tap0, u.tb_b, h->tbias, 1, 1, 0, u.tb_total, 0, R, s)))
      return rc;
  } else if ((rc = unet_time_bias(h, cond, t, R, s))) return rc;
  BlkStash* b = st->blk;
  if ((rc = block_fwd(h, 0, x, D, nullptr, 0, T, R, s))) return rc;
  if ((rc = block_fwd(h, 1, b[0].OUT, d0, nullptr, 0, T, R, s))) return rc;
  if ((rc = conv_fwd(h, u.down[0], b[1].OUT, d0, nullptr, 0, T, st->p0, T2, T2, 2, 1, 0, kOff3, u.down[0].b, R, s))) return rc;
  if ((rc = block_fwd(h, 2, st->p0, d0, nullptr, 0, T2, R, s))) return rc;
  if ((rc = block_fwd(h, 3, b[2].OUT, d1, nullptr, 0, T2, R, s))) return rc;
  if ((rc = conv_fwd(h, u.down[1], b[3].OUT, d1, nullptr, 0, T2, st->p1, T4, T4, 2, 1, 0, kOff3, u.down[1].b, R, s))) return rc;
  if ((rc = block_fwd(h, 4, st->p1, d1, nullptr, 0, T4, R, s))) return rc;
  if ((rc = block_fwd(h, 5, b[4].OUT, d2, nullptr, 0, T4, R, s))) return rc;
  if ((rc = block_fwd(h, 6, b[5].OUT, d2, nullptr, 0, T4, R, s))) return rc;
  if ((rc = block_fwd(h, 7, b[6].OUT, d2, nullptr, 0, T4, R, s))) return rc;
  if ((rc = block_fwd(h, 8, b[7].OUT, d2, b[5].OUT, d2, T4, R, s))) return rc;
  if ((rc = block_fwd(h, 9, b[8].OUT, d1, nullptr, 0, T4, R, s))) return rc;
  const int off_e[5] = {0, -1, 0, 0, 0}, off_o[5] = {1, 0, 0, 0, 0};
  if ((rc = conv_fwd(h, u.up[0][0], b[9].OUT, d1, nullptr, 0, T4, st->q0, T2, T4, 1, 2, 0, off_e, u.up_b[0], R, s))) return rc;
  if ((rc = conv_fwd(h, u.up[0][1], b[9].OUT, d1, nullptr, 0, T4, st->q0, T2, T4, 1, 2, 1, off_o, u.up_b[0], R, s))) return rc;
  if ((rc = block_fwd(h, 10, st->q0, d1, b[3].OUT, d1, T2, R, s))) return rc;
  if ((rc = block_fwd(h, 11, b[10].OUT, d0, nullptr, 0, T2, R, s))) return rc;
  if ((rc = conv_fwd(h, u.up[1][0], b[11].OUT, d0, nullptr, 0, T2, st->q1, T, T2, 1, 2, 0, off_e, u.up_b[1], R, s))) return rc;
  if ((rc = conv_fwd(h, u.up[1][1], b[11].OUT, d0, nullptr, 0, T2, st->q1, T, T2, 1, 2, 1, off_o, u.up_b[1], R, s))) return rc;
  if ((rc = conv_fwd(h, u.fin0, st->q1, d0, nullptr, 0, T, st->fA, T, T, 1, 1, 0, kOff5, u.fin0.b, R, s))) return rc;
  if ((rc = gn_mish_train(h, st->fA, u.fin0n, nullptr, 0, nullptr, st->fB, T, d0, R, s))) return rc;
  if ((rc = conv_fwd(h, u.fin1, st->fB, d0, nullptr, 0, T, eps, T, T, 1, 1, 0, kOff1, u.fin1.b, R, s))) return rc;
  st->x = x; st->t = t; st->R = R; st->fwd_valid = true;
  return 0;
}

// gradient of GroupNorm+Mish: dA = d(conv output); gamma / beta gradients -> grads; optional time-bias gradient slice
// *dA_out = this GroupNorm's own dA buffer (read later by the data gradient on `s` and by the weight gradient on the second stream)
static int gn_bwd(CldHandle* h, const float* A, const GnW& n, const float* dY, float** dA_out, float* dgamma, float* dbeta, float* dconv_bias,
                  float* dtb, int T, int C, int R, cudaStream_t s) {
  TrainState* st = ts_of(h);
  if (st->unit >= TrainState::MAX_UNITS) return fail(h, CLD_ERR_STATE, "internal: GroupNorm backward units exhausted");
  float* dA = st->gA_u[st->unit];
  float* rp = st->rp_u[st->unit];
  ++st->unit;
  *dA_out = dA;
  if (R <= 2 * h->num_sms) gn_mish_bwd_kernel<2><<<R, 512, 0, s>>>(A, n.g, n.b, dY, dA, rp, dtb, h->unet.tb_total, T, C);
  else gn_mish_bwd_kernel<1><<<R, 256, 0, s>>>(A, n.g, n.b, dY, dA, rp, dtb, h->unet.tb_total, T, C);
  CLD_LAUNCH_OK(h, "gn_mish_bwd_kernel");
  return colsum(h, rp, R, 3 * C, dgamma, pg_stream(h, s), C, dbeta, dconv_bias);
}

static const int kK5[5] = {0, 1, 2, 3, 4}, kK1[5] = {0, 0, 0, 0, 0}, kK3[5] = {0, 1, 2, 0, 0};
static const int kTap5[5] = {0, 1, 2, 3, 4};
static const int kNeg5[5] = {2, 1, 0, -1, -2};

// weight + bias gradient of a stride-1 convolution with `ntaps` (5 | 1) taps
static int conv_param_grads(CldHandle* h, int cin_total, int cout, int ntaps, const float* in0, int c0, const float* in1, int c1, int T,
                            const float* dout, float* dw, float* db, int R, cudaStream_t s) {
  int rc, splits;
  // db == nullptr: the bias gradient came out of the GroupNorm backward that produced `dout`
  bool bias_in_part;
  s = pg_stream(h, s);
  if ((rc = conv_wgrad(h, cin_total, cout, ntaps, ntaps == 5 ? kOff5 : kOff1, in0, c0, in1, c1, T, dout, T, T, 1, 1, 0, R, &splits, s,
                       db != nullptr, &bias_in_part)))
    return rc;
  if ((rc = wreduce(h, splits, ntaps, cin_total, cout, 0, cout, dw, ntaps, ntaps == 5 ? kK5 : kK1, 0, s, bias_in_part ? db : nullptr))) return rc;
  return (db && !bias_in_part) ? colsum(h, dout, R * T, cout, db, s) : 0;
}

// backward of one residual block.  dOUT [R,T,cout] -> dIN [R,T,cin_total] (written), parameter gradients -> grads[...]
static int block_bwd(CldHandle* h, int bi, const BlkIdx& ix, const float* dOUT, float* dIN, float* const* grads, int R, cudaStream_t s) {
  TrainState* st = ts_of(h);
  const ResBlockW& rb = h->unet.rb[bi];
  const BlkStash& b = st->blk[bi];
  const int T = b.T, C = rb.cout, cin = b.c0 + b.c1;
  int rc;
  // second Conv1dBlock
  float* gA;
  if ((rc = gn_bwd(h, b.A1, rb.n1, dOUT, &gA, grads[ix.g1], grads[ix.b1], grads[ix.c1b], nullptr, T, C, R, s))) return rc;
  if ((rc = conv_param_grads(h, C, C, 5, b.B0, C, nullptr, 0, T, gA, grads[ix.c1w], nullptr, R, s))) return rc;
  if ((rc = conv_dgrad(h, rb.c1, 5, kTap5, kNeg5, gA, T, st->gB, T, C, T, 1, 1, 0, 0, R, s))) return rc;
  // first Conv1dBlock (+ time / cond bias)
  if ((rc = gn_bwd(h, b.A0, rb.n0, st->gB, &gA, grads[ix.g0], grads[ix.b0], grads[ix.c0b], st->dtbias + rb.tb_off, T, C, R, s))) return rc;
  if ((rc = conv_param_grads(h, cin, C, 5, b.in0, b.c0, b.in1, b.c1, T, gA, grads[ix.c0w], nullptr, R, s))) return rc;
  if ((rc = conv_dgrad(h, rb.c0, 5, kTap5, kNeg5, gA, T, dIN, T, cin, T, 1, 1, 0, 0, R, s))) return rc;
  // residual path
  if (rb.res.w) {
    if ((rc = conv_param_grads(h, cin, C, 1, b.in0, b.c0, b.in1, b.c1, T, dOUT, grads[ix.rw], grads[ix.rb], R, s))) return rc;
    const int tap0[5] = {0, 0, 0, 0, 0};
    if ((rc = conv_dgrad(h, rb.res, 1, tap0, kOff1, dOUT, T, dIN, T, cin, T, 1, 1, 0, 1, R, s))) return rc;
  } else {
    if ((rc = slice(h, dIN, dOUT, (size_t)R * T, C, C, 0, 1, s))) return rc;
  }
  return 0;
}

// backward of Downsample1d (Conv1d k3 s2 p1): in [R,T,C] -> out [R,T/2,C]
static int down_bwd(CldHandle* h, const ConvW& w, const float* in, int T, const float* dout, float* din, float* dw, float* db, int R,
                    cudaStream_t s) {
  const int C = w.cout, Th = T / 2;
  int rc, splits;
  bool bias_in_part;
  cudaStream_t ps = pg_stream(h, s);
  if ((rc = conv_wgrad(h, C, C, 3, kOff3, in, C, nullptr, 0, T, dout, Th, Th, 2, 1, 0, R, &splits, ps, true, &bias_in_part))) return rc;
  if ((rc = wreduce(h, splits, 3, C, C, 0, C, dw, 3, kK3, 0, ps, bias_in_part ? db : nullptr))) return rc;
  if (!bias_in_part && (rc = colsum(h, dout, R * Th, C, db, ps))) return rc;
  // forward: out[j] = sum_tap in[2j + tap - 1] W[tap].  even ti = 2m: tap 1, j = m;  odd ti = 2m + 1: tap 0 with j = m + 1, tap 2 with j = m
  const int te[5] = {1, 0, 0, 0, 0}, oe[5] = {0, 0, 0, 0, 0};
  const int to[5] = {0, 2, 0, 0, 0}, oo[5] = {1, 0, 0, 0, 0};
  if ((rc = conv_dgrad(h, w, 1, te, oe, dout, Th, din, T, C, Th, 1, 2, 0, 0, R, s))) return rc;
  return conv_dgrad(h, w, 2, to, oo, dout, Th, din, T, C, Th, 1, 2, 1, 0, R, s);
}

// backward of Upsample1d (ConvTranspose1d k4 s2 p1): in [R,T,C] -> out [R,2T,C]; phases packed as up[0] (even outputs: torch taps 1, 3
// reading in[j], in[j-1]) and up[1] (odd outputs: torch taps 0, 2 reading in[j+1], in[j])
static int up_bwd(CldHandle* h, const ConvW* up, const float* in, int T, const float* dout, float* din, float* dw, float* db, int R,
                  cudaStream_t s) {
  const int C = up[0].cout;
  const int off_e[5] = {0, -1, 0, 0, 0}, off_o[5] = {1, 0, 0, 0, 0};
  const int kte[5] = {1, 3, 0, 0, 0}, kto[5] = {0, 2, 0, 0, 0};
  int rc, splits;
  cudaStream_t ps = pg_stream(h, s);
  if ((rc = conv_wgrad(h, C, C, 2, off_e, in, C, nullptr, 0, T, dout, 2 * T, T, 1, 2, 0, R, &splits, ps))) return rc;
  if ((rc = wreduce(h, splits, 2, C, C, 0, C, dw, 4, kte, 1, ps))) return rc;
  if ((rc = conv_wgrad(h, C, C, 2, off_o, in, C, nullptr, 0, T, dout, 2 * T, T, 1, 2, 1, R, &splits, ps))) return rc;
  if ((rc = wreduce(h, splits, 2, C, C, 0, C, dw, 4, kto, 1, ps))) return rc;
  if ((rc = colsum(h, dout, R * 2 * T, C, db, ps))) return rc;
  // dIn[ti] = sum_ph sum_tap dOut[2 (ti - io_ph[tap]) + ph] W_ph[tap]^T
  const int t01[5] = {0, 1, 0, 0, 0};
  const int ie[5] = {0, 2, 0, 0, 0};          // phase 0: -2 * {0, -1} + 0
  const int io[5] = {-1, 1, 0, 0, 0};         // phase 1: -2 * {1, 0} + 1
  if ((rc = conv_dgrad(h, up[0], 2, t01, ie, dout, 2 * T, din, T, C, T, 2, 1, 0, 0, R, s))) return rc;
  return conv_dgrad(h, up[1], 2, t01, io, dout, 2 * T, din, T, C, T, 2, 1, 0, 1, R, s);
}

int unet_train_backward(CldHandle* h, const float* d_eps, float* const* grads, int n, float* dx_out, int R, cudaStream_t s) {
  TrainState* st = ts_of(h);
  if (!st || !st->fwd_valid || st->R != R)
    return fail(h, CLD_ERR_STATE, "cld_unet_backward needs the cld_unet_train_forward of the same rows immediately before it");
  const UnetW& u = h->unet;
  const CldConfig& c = h->cfg;
  const int T = c.horizon, T2 = T / 2, T4 = T / 4;
  const int d0 = c.dims[0], d1 = c.dims[1], d2 = c.dims[2], D = c.latent_dim, td = c.base_dim, tdim = c.base_dim + c.cond_dim;
  const UnetLayout& L = h->unet_layout;
  if (n != (int)L.numel.size()) return fail(h, CLD_ERR_ARG, "cld_unet_backward: expected %zu gradient tensors, got %d", L.numel.size(), n);
  const BlkIdx* ix = L.blk;
  int rc, splits;
  const BlkStash* b = st->blk;
  st->unit = 0; st->nd = 0;
  auto nb = [&]() -> float* { return st->gD[st->nd < TrainState::MAX_GD ? st->nd++ : TrainState::MAX_GD - 1]; };   // a fresh data-gradient buffer
  float *g, *g2, *gA;
  // ---- final_conv: Conv1d(1x1) <- Conv1dBlock
  if ((rc = conv_param_grads(h, d0, D, 1, st->fB, d0, nullptr, 0, T, d_eps, grads[L.fin[4]], grads[L.fin[5]], R, s))) return rc;
  g = nb();
  {
    const int tap0[5] = {0, 0, 0, 0, 0};
    if ((rc = conv_dgrad(h, u.fin1, 1, tap0, kOff1, d_eps, T, g, T, d0, T, 1, 1, 0, 0, R, s))) return rc;
  }
  if ((rc = gn_bwd(h, st->fA, u.fin0n, g, &gA, grads[L.fin[2]], grads[L.fin[3]], grads[L.fin[1]], nullptr, T, d0, R, s))) return rc;
  if ((rc = conv_param_grads(h, d0, d0, 5, st->q1, d0, nullptr, 0, T, gA, grads[L.fin[0]], nullptr, R, s))) return rc;
  g = nb();
  if ((rc = conv_dgrad(h, u.fin0, 5, kTap5, kNeg5, gA, T, g, T, d0, T, 1, 1, 0, 0, R, s))) return rc;               // g = d q1
  // ---- ups.1: upsample, blocks 11, 10
  g2 = nb();
  if ((rc = up_bwd(h, u.up[1], b[11].OUT, T2, g, g2, grads[L.up[1][0]], grads[L.up[1][1]], R, s))) return rc;       // g2 = d o11
  g = nb();
  if ((rc = block_bwd(h, 11, ix[11], g2, g, grads, R, s))) return rc;                                               // g = d o10
  if ((rc = block_bwd(h, 10, ix[10], g, st->gcat10, grads, R, s))) return rc;                                       // (d q0 | d sk1)
  g = nb();
  if ((rc = slice(h, g, st->gcat10, (size_t)R * T2, d1, 2 * d1, 0, 0, s))) return rc;                               // g = d q0
  // ---- ups.0: upsample, blocks 9, 8
  g2 = nb();
  if ((rc = up_bwd(h, u.up[0], b[9].OUT, T4, g, g2, grads[L.up[0][0]], grads[L.up[0][1]], R, s))) return rc;        // g2 = d o9
  g = nb();
  if ((rc = block_bwd(h, 9, ix[9], g2, g, grads, R, s))) return rc;                                                 // g = d o8
  if ((rc = block_bwd(h, 8, ix[8], g, st->gcat8, grads, R, s))) return rc;                                          // (d o7 | d sk2)
  g = nb();
  if ((rc = slice(h, g, st->gcat8, (size_t)R * T4, d2, 2 * d2, 0, 0, s))) return rc;                                // g = d o7
  // ---- mid blocks 7, 6
  g2 = nb();
  if ((rc = block_bwd(h, 7, ix[7], g, g2, grads, R, s))) return rc;                                                 // g2 = d o6
  g = nb();
  if ((rc = block_bwd(h, 6, ix[6], g2, g, grads, R, s))) return rc;                                                 // g = d o5 (mid part)
  if ((rc = slice(h, g, st->gcat8, (size_t)R * T4, d2, 2 * d2, d2, 1, s))) return rc;                               // + skip part
  // ---- downs.2: blocks 5, 4
  g2 = nb();
  if ((rc = block_bwd(h, 5, ix[5], g, g2, grads, R, s))) return rc;                                                 // g2 = d o4
  g = nb();
  if ((rc = block_bwd(h, 4, ix[4], g2, g, grads, R, s))) return rc;                                                 // g = d p1
  // ---- downs.1: downsample, blocks 3, 2
  g2 = nb();
  if ((rc = down_bwd(h, u.down[1], b[3].OUT, T2, g, g2, grads[L.down[1][0]], grads[L.down[1][1]], R, s))) return rc;    // g2 = d o3 (down part)
  if ((rc = slice(h, g2, st->gcat10, (size_t)R * T2, d1, 2 * d1, d1, 1, s))) return rc;                             // + skip part
  g = nb();
  if ((rc = block_bwd(h, 3, ix[3], g2, g, grads, R, s))) return rc;                                                 // g = d o2
  g2 = nb();
  if ((rc = block_bwd(h, 2, ix[2], g, g2, grads, R, s))) return rc;                                                 // g2 = d p0
  // ---- downs.0: downsample, blocks 1, 0
  g = nb();
  if ((rc = down_bwd(h, u.down[0], b[1].OUT, T, g2, g, grads[L.down[0][0]], grads[L.down[0][1]], R, s))) return rc;     // g = d o1
  g2 = nb();
  if ((rc = block_bwd(h, 1, ix[1], g, g2, grads, R, s))) return rc;                                                 // g2 = d o0
  g = nb();
  if ((rc = block_bwd(h, 0, ix[0], g2, g, grads, R, s))) return rc;                                                 // g = d x [R,T,4]
  if (dx_out) CLD_CUDA_OK(h, cudaMemcpyAsync(dx_out, g, (size_t)R * T * D * sizeof(float), cudaMemcpyDeviceToDevice, s));
  // ---- time / cond projections of the 12 blocks: tbias = tcm @ tb_w + tb_b  (tb_w packed [tdim][tb_total]); everything from here
  //      on is parameter-gradient work: on the second stream, after the last GroupNorm backward has written its slice of dtbias
  cudaStream_t ps = pg_stream(h, s);
  const int tbt = u.tb_total;
  if ((rc = conv_wgrad(h, tdim, tbt, 1, kOff1, h->tcm, tdim, nullptr, 0, 1, st->dtbias, 1, 1, 1, 1, 0, R, &splits, ps))) return rc;
  for (int e = 0; e < 12; ++e)
    if ((rc = wreduce(h, splits, 1, tdim, tbt, u.rb[e].tb_off, u.rb[e].cout, grads[ix[e].tw], 1, kK1, 0, ps))) return rc;
  if ((rc = colsum(h, st->dtbias, R, tbt, st->tb_bgrad, ps))) return rc;
  for (int e = 0; e < 12; ++e)
    CLD_CUDA_OK(h, cudaMemcpyAsync(grads[ix[e].tb], st->tb_bgrad + u.rb[e].tb_off, u.rb[e].cout * sizeof(float),
                                   cudaMemcpyDeviceToDevice, ps));
  // d(Mish(time embedding)) = dtbias @ tb_w[0:td, :]^T   (the cond half of tcm is an input, not a parameter)
  {
    ConvW tb; tb.w = u.tb_w; tb.cin = tdim; tb.cout = tbt; tb.ntaps = 1;
    const int tap0[5] = {0, 0, 0, 0, 0};
    if ((rc = conv_dgrad(h, tb, 1, tap0, kOff1, st->dtbias, 1, st->dtcm, 1, td, 1, 1, 1, 0, 0, R, ps))) return rc;
  }
  time_mlp_bwd_kernel<<<R, 128, 0, ps>>>(st->t, u.t1_w, u.t1_b, u.t2_w, u.t2_b, u.freqs, st->dtcm, td, st->emb, st->hid, st->dpre1,
                                         st->dpre2, td);
  CLD_LAUNCH_OK(h, "time_mlp_bwd_kernel");
  // Linear(d, 4d): weight [4d][d];  Linear(4d, d): weight [d][4d]
  if ((rc = conv_wgrad(h, td, 4 * td, 1, kOff1, st->emb, td, nullptr, 0, 1, st->dpre1, 1, 1, 1, 1, 0, R, &splits, ps))) return rc;
  if ((rc = wreduce(h, splits, 1, td, 4 * td, 0, 4 * td, grads[L.tmlp[0]], 1, kK1, 0, ps))) return rc;
  if ((rc = colsum(h, st->dpre1, R, 4 * td, grads[L.tmlp[1]], ps))) return rc;
  if ((rc = conv_wgrad(h, 4 * td, td, 1, kOff1, st->hid, 4 * td, nullptr, 0, 1, st->dpre2, 1, 1, 1, 1, 0, R, &splits, ps))) return rc;
  if ((rc = wreduce(h, splits, 1, 4 * td, td, 0, td, grads[L.tmlp[2]], 1, kK1, 0, ps))) return rc;
  if ((rc = colsum(h, st->dpre2, R, td, grads[L.tmlp[3]], ps))) return rc;
  pg_join(h, s);                 // the gradients are complete in the caller's stream order
  return 0;
}

static int upload_schedule(CldHandle* h, cudaStream_t s) {
  TrainState* st = ts_of(h);
  const Schedule& sc = h->sched;
  if (!sc.loaded) return fail(h, CLD_ERR_STATE, "schedule not loaded");
  const int n = h->cfg.n_timesteps;
  CLD_CUDA_OK(h, cudaMemcpyAsync(st->sched_dev, sc.x_t_cof.data(), n * sizeof(float), cudaMemcpyHostToDevice, s));
  CLD_CUDA_OK(h, cudaMemcpyAsync(st->sched_dev + n, sc.noise_cof.data(), n * sizeof(float), cudaMemcpyHostToDevice, s));
  CLD_CUDA_OK(h, cudaMemcpyAsync(st->sched_dev + 2 * n, sc.logvar.data(), n * sizeof(float), cudaMemcpyHostToDevice, s));
  return 0;
}

int ppo_head(CldHandle* h, const float* eps, const float* x_t, const float* x_tm1, const int64_t* t, const float* logp_old,
             const float* reward, float baseline, const float* baseline_dev, float clip, float* logp_new, float* loss_out, float* d_eps, int R,
             cudaStream_t s) {
  int rc;
  if ((rc = train_prepare(h, R))) return rc;
  if (ts_of(h)->sched_version != h->sched_version) {         // host -> device copy only when the schedule changed (never inside a CUDA graph)
    if ((rc = upload_schedule(h, s))) return rc;
    ts_of(h)->sched_version = h->sched_version;
  }
  TrainState* st = ts_of(h);
  const int n = h->cfg.horizon * h->cfg.latent_dim;
  ppo_head_kernel<<<R, 128, 0, s>>>(eps, x_t, x_tm1, t, st->sched_dev, h->cfg.n_timesteps, logp_old, reward, baseline, baseline_dev, clip, logp_new,
                                    st->loss_row, d_eps, n, R);
  CLD_LAUNCH_OK(h, "ppo_head_kernel");
  if (loss_out) {
    sum_rows_kernel<<<1, 256, 0, s>>>(st->loss_row, R, loss_out);
    CLD_LAUNCH_OK(h, "sum_rows_kernel");
  }
  return 0;
}

int mse_head(CldHandle* h, const float* eps, const float* noise, float* loss_out, float* d_eps, int R, cudaStream_t s) {
  int rc;
  if ((rc = train_prepare(h, R))) return rc;
  TrainState* st = ts_of(h);
  const int n = h->cfg.horizon * h->cfg.latent_dim;
  mse_head_kernel<<<R, 128, 0, s>>>(eps, noise, st->loss_row, d_eps, n, R);
  CLD_LAUNCH_OK(h, "mse_head_kernel");
  if (loss_out) {
    sum_rows_kernel<<<1, 256, 0, s>>>(st->loss_row, R, loss_out);
    CLD_LAUNCH_OK(h, "sum_rows_kernel");
  }
  return 0;
}

float* train_deps_buffer(CldHandle* h) { return ts_of(h) ? ts_of(h)->deps : nullptr; }

int adam_step(CldHandle* h, float* p, const float* g, float* m, float* v, size_t n, double lr, double b1, double b2, double eps, double wd,
              int step, cudaStream_t s) {
  // the scalar factors in double, as torch's Python-side arithmetic computes them (1 - 0.999f evaluated in fp32 is off by 1.3e-5)
  const float step_size = (float)(lr / (1.0 - pow(b1, (double)step)));
  const float bc2_sqrt = (float)sqrt(1.0 - pow(b2, (double)step));
  adam_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(p, g, m, v, n, step_size, (float)(1.0 - b1), (float)b2, (float)(1.0 - b2), (float)eps,
                                                          (float)wd, bc2_sqrt, nullptr);
  CLD_LAUNCH_OK(h, "adam_kernel");
  return 0;
}

int adam_step_dev(CldHandle* h, float* p, const float* g, float* m, float* v, size_t n, const double* lr_dev, long long* step_dev, double b1,
                  double b2, double eps, double wd, cudaStream_t s) {
  int rc;
  if ((rc = train_prepare(h, 1))) return rc;
  TrainState* st = ts_of(h);
  adam_tick_kernel<<<1, 1, 0, s>>>(step_dev, lr_dev, b1, b2, st->adam_dyn);
  CLD_LAUNCH_OK(h, "adam_tick_kernel");
  adam_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(p, g, m, v, n, 0.f, (float)(1.0 - b1), (float)b2, (float)(1.0 - b2), (float)eps, (float)wd,
                                                          1.f, st->adam_dyn);
  CLD_LAUNCH_OK(h, "adam_kernel");
  return 0;
}

}  // namespace cld
