// LSTM decoder on the tensor pipe (bf16-precision mode): forward + rollout, and the analytic backward (BPTT).
//   Decoder.forward                         reference models/vae/lstm_vae.py:44-52
//   convert_action_to_state_and_action      reference models/vae/vae_model.py:100-129,157-173
//   unicyle_forward_dynamics('parallel')    reference src/tbsim/models/diffuser_helpers.py:573-639
//   PerturbationGuidance.perturb (backward) reference src/tbsim/utils/guidance_loss.py:2250-2278
//
// One CTA owns 32 rows for the whole horizon.  Per time step and layer the gate pre-activations are
//   gates^T [256 x 32 rows] = W [256 x K] . [x_t ; h_{t-1}]^T [K x 32]
// i.e. the WEIGHTS are the M operand (two M = 128 tiles, resident in shared memory as fp16, 128B-swizzled) and
// the 32 rows are the N operand, so a CTA needs only 32 rows to fill a tile and 4 096 rows spread over 128 SMs.
// The state operand is written by the cell warps as an fp16 hi + lo pair (two accumulating MMA passes): the
// activations carry ~22 mantissa bits, the weights are rounded to fp16 once (the backward uses the same rounded
// weights, so it is the exact gradient of the model the forward evaluates).  Accumulators live in TMEM
// (4 x 32 columns); a cell thread reads ITS lane = one gate row for all 32 rows.  Gate rows are permuted so that
// lanes j and j + 16 of a warp hold (i, g) and (f, o) of the same hidden unit: the two exchange what they need with
// warp shuffles, then each updates the cell for 16 of the 32 rows -- no shared-memory exchange, uniform code.
// The two layers run skewed by one step on separate warp sets; everything is synchronised with mbarriers
// (MMA completion -> cell warps -> operand ready -> MMA issue).
//
// Warp roles (576 threads): warps 0-7 layer-0 cells, warps 8-15 layer-1 cells (warp & 3 = TMEM lane quadrant,
// (warp >> 2) & 1 = row half), warp 16 MMA issuer (event loop, one issuing thread), warp 17: stages z_t as an MMA
// operand, hid2act and the unicycle rollout step by step (lane = row).
#include <cuda_fp16.h>
#include <stdio.h>
#include <stdlib.h>

#include "common.cuh"
#include "lstm_shared.cuh"
#include "tc_common.cuh"

namespace cld {
using namespace tc;

namespace {
constexpr int LT_RB = 32;                 // rows per CTA = MMA N
constexpr int LT_H = 64;
constexpr int LT_THREADS = 576;
constexpr int LT_WBLK = 16384;            // one weight k-block: 128 gate rows x 64 k fp16
constexpr int LT_OP = 4096;               // one state operand tile: 32 rows x 64 k fp16
// forward kernel shared memory (bytes from the 1024-aligned base)
constexpr int LF_H0 = 0;                              // h0 operand [parity][hi, lo]
constexpr int LF_H1 = LF_H0 + 4 * LT_OP;              // h1 operand [hi, lo]
constexpr int LF_Z = LF_H1 + 2 * LT_OP;               // z operand [ring of 3][hi, lo] (k 0..3 used)
constexpr int LF_H1F = LF_Z + 6 * LT_OP;              // fp32 h1 [parity][32 rows][65] for hid2act (row pitch 65: conflict-free both ways)
constexpr int LF_H1P = LT_H + 1;
constexpr int LF_HW = LF_H1F + 2 * LT_RB * LF_H1P * 4;  // hid2act weights [2][64]
constexpr int LF_BARS = LF_HW + 2 * LT_H * 4;         // m0, m1, e0, e1, a, z[3]
constexpr int LF_TMEM = LF_BARS + 8 * 8;
constexpr int LF_SMEM = LF_TMEM + 16;
static_assert(LF_SMEM + 1024 <= 232448, "forward shared memory");

constexpr int LF_WCOL0 = 192, LF_WCOLS = 208;        // forward weights in TMEM: columns [192, 400)
constexpr int LB_WCOL0 = 192, LB_WCOLS = 256;        // backward weights in TMEM: columns [192, 448)

constexpr int LT_MIN_SMEM = 120 * 1024;              // requested at least: one CTA per SM (each CTA allocates all 512 TMEM columns)

constexpr float LOG2E = 1.4426950408889634f;

__host__ __device__ constexpr uint32_t idesc_f16(int M, int N) {
  return (1u << 4) | (1u << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);      // D fp32, A/B fp16, A K-major (TMEM), B N-major
}
__device__ __forceinline__ float ex2f(float x) { float r; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float rcpf(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
// s * sigmoid(-k x / log2e) + o  with (k, s, o) = (-log2e, 1, 0): sigmoid(x) ; (-2 log2e, 2, -1): tanh(x)
__device__ __forceinline__ float act_gen(float x, float k, float s, float o) { return fmaf(s, rcpf(1.0f + ex2f(k * x)), o); }
__device__ __forceinline__ float sigmoidf_(float x) { return rcpf(1.0f + ex2f(-LOG2E * x)); }
__device__ __forceinline__ float tanhf_(float x) { return fmaf(2.0f, rcpf(1.0f + ex2f(-2.0f * LOG2E * x)), -1.0f); }

// D[tmem] (+)= A[tmem] * B[smem]^T : the A operand (here: the LSTM weights, resident for the whole kernel) is read
// from tensor memory -- lane = M row, one 32-bit column = two consecutive K elements (fp16x2, low half = even k).
// With N = 32 an SS-mode MMA is bound by the 4 KB A fetch from shared memory (62 cycles measured); the TS form takes
// 17 cycles (tools/umma_ts_bench.cu).
__device__ __forceinline__ void umma_ts_f16(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// weights -> TMEM: `blob` is [ncols][128 lanes] uint32 (fp16x2); the 4 warps of each lane quadrant take the 8-column chunks round robin
__device__ __forceinline__ void load_weights_tmem(const uint32_t* __restrict__ blob, int ncols, uint32_t tmem_col0, int q, int rq, int lane) {
  for (int chunk = rq; chunk * 8 < ncols; chunk += 4) {
    uint32_t r[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) r[c] = blob[(size_t)(chunk * 8 + c) * 128 + q * 32 + lane];
    tmem_st8(tmem_col0 + ((uint32_t)(q * 32) << 16) + (uint32_t)(chunk * 8), r);
  }
  tmem_wait_st();
}

// mbarrier wait with a watchdog: a protocol bug traps (launch error) instead of hanging the device
__device__ __noinline__ void lt_wait_timeout(uint32_t bar, uint32_t parity, int tag) {
  const long long t0 = clock64();
  bool said = false;
  while (!mbar_try_wait(bar, parity)) {
    const long long dt = clock64() - t0;
    if (dt > 2000000000ll && !said) {
      said = true;
      if ((threadIdx.x & 31) == 0)
        printf("lstm_tc: mbarrier wait timed out (tag %d, block %d, warp %d, parity %u)\n", tag, (int)blockIdx.x, (int)(threadIdx.x >> 5), parity);
    }
    if (dt > 4000000000ll) __trap();
  }
}
__device__ __forceinline__ void lt_wait(uint32_t bar, uint32_t parity, int tag) {
  if (!mbar_try_wait(bar, parity)) lt_wait_timeout(bar, parity, tag);
}

// State operand tiles (MMA N operand: 32 rows x 64 k, fp16) are N-MAJOR: 64-byte lines of the 32 rows for one k, 64-byte
// swizzle (16-byte chunk index ^= (k >> 1) & 3), 8 k per 512-byte atom.  A cell thread owns one k (its hidden unit) and 8
// consecutive rows, i.e. exactly one 16-byte chunk: one STS.128 per tile instead of eight 2-byte stores.  Descriptor: SBO = 512,
// layout SWIZZLE_64B, one K = 16 step = 1024 bytes; instruction descriptor bit 16 (B is MN-major).  (Probed on hardware:
// tools/umma_ts_bench.cu.)
__host__ __device__ constexpr uint32_t nmaj_off(uint32_t n, uint32_t k) { return k * 64u + ((((n >> 3) ^ (k >> 1)) & 3u) << 4) + (n & 7u) * 2u; }
__device__ __forceinline__ uint64_t make_desc_nmaj(uint32_t smem_addr) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(512 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)4 << 61);
}
constexpr int NMAJ_KSTEP = 1024 >> 4;      // descriptor units (16 bytes) per K = 16 step

// fp16 hi/lo split of v (lo = (v - hi) * lo_scale), stored at element (row n, k) of the operand tiles `hi` and `hi + LT_OP`
__device__ __forceinline__ void store_split(uint8_t* hi, int row, int k, float v, float lo_scale = 1.0f) {
  const __half h = __float2half_rn(v);
  const __half l = __float2half_rn((v - __half2float(h)) * lo_scale);
  const uint32_t off = nmaj_off((uint32_t)row, (uint32_t)k);
  *reinterpret_cast<__half*>(hi + off) = h;
  *reinterpret_cast<__half*>(hi + LT_OP + off) = l;
}
// the same for 8 consecutive rows (row block rb) of one k: two 16-byte stores
__device__ __forceinline__ void store_split8(uint8_t* hi, int rb, int k, const float (&v)[8], float lo_scale = 1.0f, int lo_off = LT_OP) {
  uint32_t ph[4], pl[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const __half2 h = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
    const float2 hf = __half22float2(h);
    const __half2 l = __floats2half2_rn((v[2 * i] - hf.x) * lo_scale, (v[2 * i + 1] - hf.y) * lo_scale);
    ph[i] = *reinterpret_cast<const uint32_t*>(&h);
    pl[i] = *reinterpret_cast<const uint32_t*>(&l);
  }
  const uint32_t off = (uint32_t)k * 64u + ((((uint32_t)rb ^ ((uint32_t)k >> 1)) & 3u) << 4);
  *reinterpret_cast<uint4*>(hi + off) = make_uint4(ph[0], ph[1], ph[2], ph[3]);
  *reinterpret_cast<uint4*>(hi + lo_off + off) = make_uint4(pl[0], pl[1], pl[2], pl[3]);
}

// gate row held by lane m (0..127) of M tile `tile`: lanes j, j + 16 of quadrant q serve unit 16 q + j
__host__ __device__ inline int gate_row_of(int tile, int m) {
  const int q = m >> 5, l = m & 31, j = l & 15, is_b = l >> 4, u = 16 * q + j;
  const int gate = tile == 0 ? (is_b ? 1 : 0) : (is_b ? 3 : 2);      // nn.LSTM order i, f, g, o
  return gate * LT_H + u;
}
}  // namespace

// 32-byte stash accesses (LDG/STG.256): one full sector per instruction
__device__ __forceinline__ void st8(float* p, float v0, float v1, float v2, float v3, float v4, float v5, float v6, float v7) {
  asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               :: "l"(p), "f"(v0), "f"(v1), "f"(v2), "f"(v3), "f"(v4), "f"(v5), "f"(v6), "f"(v7) : "memory");
}
struct LstmTcArgs {
  const float *z, *h0, *curr;
  const uint8_t* wblob;                  // packed fp16x2 forward weights for TMEM, [208][128]
  const float *b0, *b1;                  // b_ih + b_hh per layer [256]
  const float *h2a_w, *h2a_b;
  float *act_out, *traj_out, *stash;
  int R, T;
  DynParams2 dyn;
};

// forward weight blob for TMEM: [208 columns][128 lanes] fp16x2 (two consecutive k per column).  Columns: layer 0 tile t at 40 t
// (W_hh0: 32 columns, then W_ih0: k < 4 of a K = 16 step, rest zero); layer 1 tile t at 80 + 64 t (W_ih1: 32 columns, W_hh1: 32).
__global__ void lstm_tc_pack_fwd_kernel(uint32_t* __restrict__ out, const float* __restrict__ wih0, const float* __restrict__ whh0,
                                        const float* __restrict__ wih1, const float* __restrict__ whh1) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= LF_WCOLS * 128) return;
  const int m = idx & 127, c = idx >> 7;
  float v0, v1;
  if (c < 80) {
    const int tile = c / 40, cc = c % 40, row = gate_row_of(tile, m);
    if (cc < 32) { v0 = whh0[row * 64 + 2 * cc]; v1 = whh0[row * 64 + 2 * cc + 1]; }
    else { const int k = 2 * (cc - 32); v0 = k < 4 ? wih0[row * 4 + k] : 0.f; v1 = k + 1 < 4 ? wih0[row * 4 + k + 1] : 0.f; }
  } else {
    const int tile = (c - 80) / 64, cc = (c - 80) % 64, row = gate_row_of(tile, m);
    const float* w = cc < 32 ? wih1 : whh1;
    const int k = 2 * (cc & 31);
    v0 = w[row * 64 + k]; v1 = w[row * 64 + k + 1];
  }
  const __half2 h = __floats2half2_rn(v0, v1);
  out[idx] = *reinterpret_cast<const uint32_t*>(&h);
}

template <bool SAVE, bool PROF>
__global__ void __launch_bounds__(LT_THREADS, 1) lstm_decode_tc_kernel(const LstmTcArgs a) {
  constexpr int P0 = 20, PN = 4;        // CLD_LSTM_PROF=1: timeline of steps P0 .. P0+PN-1 of CTA 0 (clock64), printed at the end
  long long tl[PN][6];
  const bool rec = PROF && blockIdx.x == 0 && (threadIdx.x & 31) == 0;
  const long long tbase = PROF ? clock64() : 0;
  (void)tl; (void)rec; (void)tbase;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* sm = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int row0 = blockIdx.x * LT_RB, T = a.T, R = a.R;
  const uint32_t bars = smem_u32(sm + LF_BARS);
  const uint32_t bar_m0 = bars, bar_m1 = bars + 8, bar_e0 = bars + 16, bar_e1 = bars + 24, bar_a = bars + 32, bar_z = bars + 40;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm + LF_TMEM);
  float* h1f = reinterpret_cast<float*>(sm + LF_H1F);
  float* hw = reinterpret_cast<float*>(sm + LF_HW);

  // ---- prologue: weights, zeroed operand tiles, initial state h_{-1} = cond2hidden(cond) for both layers
  {
    uint4* ops = reinterpret_cast<uint4*>(sm + LF_H0);
    for (int i = tid; i < (LF_H1F - LF_H0) / 16; i += LT_THREADS) ops[i] = make_uint4(0u, 0u, 0u, 0u);
    if (tid < 2 * LT_H) hw[tid] = a.h2a_w[tid];
    if (tid == 0) {
      mbar_init(bar_m0, 1); mbar_init(bar_m1, 1); mbar_init(bar_e0, 8); mbar_init(bar_e1, 8); mbar_init(bar_a, 1);
      mbar_init(bar_z, 1); mbar_init(bar_z + 8, 1); mbar_init(bar_z + 16, 1);
      fence_barrier_init();
    }
  }
  __syncthreads();
  for (int i = tid; i < LT_RB * LT_H; i += LT_THREADS) {
    const int rl = i >> 6, k = i & 63;
    const float v = (row0 + rl < R) ? a.h0[(size_t)(row0 + rl) * LT_H + k] : 0.f;
    store_split(sm + LF_H0 + 2 * LT_OP, rl, k, v);          // parity 1 = step -1
    store_split(sm + LF_H1, rl, k, v);
  }
  if (warp == 17) {                                          // z_0, z_1, z_2
    for (int t = 0; t < 3 && t < T; ++t) {
      float4 zv = make_float4(0.f, 0.f, 0.f, 0.f);
      if (row0 + lane < R) zv = reinterpret_cast<const float4*>(a.z)[(size_t)(row0 + lane) * T + t];
      uint8_t* zt = sm + LF_Z + t * 2 * LT_OP;
      store_split(zt, lane, 0, zv.x); store_split(zt, lane, 1, zv.y); store_split(zt, lane, 2, zv.z); store_split(zt, lane, 3, zv.w);
    }
  }
  if (warp == 16) { tmem_alloc(smem_u32(tmem_slot), 512); tmem_relinquish(); }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (warp < 16) load_weights_tmem(reinterpret_cast<const uint32_t*>(a.wblob), LF_WCOLS, tmem_base + LF_WCOL0, warp & 3, warp >> 2, lane);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  // TMEM columns: layer 0 [tile 0 | tile 1] at 0..63 ; layer 1 [step parity][tile 0 | tile 1] at 64..191 ;
  // weights (A operand) at 192..399: layer 0 [tile][W_hh0 32 | W_ih0 8], then layer 1 [tile][W_ih1 32 | W_hh1 32]

  if (warp < 16) {
    // ===================== cell warps: (layer, lane quadrant, row half) =====================
    const int L = warp >> 3, q = warp & 3, rh = (warp >> 2) & 1, j = lane & 15;
    const bool is_b = lane >= 16;
    const int u = 16 * q + j;
    const uint32_t lane_t = tmem_base + ((uint32_t)(q * 32) << 16);
    const float* bias = L == 0 ? a.b0 : a.b1;
    const float bias0 = bias[(is_b ? 64 : 0) + u];            // tile 0: i | f
    const float bias1 = bias[(is_b ? 192 : 128) + u];         // tile 1: g | o
    const float k1 = is_b ? -LOG2E : -2.0f * LOG2E, s1c = is_b ? 1.0f : 2.0f, o1c = is_b ? 0.0f : -1.0f;
    const uint32_t bar_m = L == 0 ? bar_m0 : bar_m1, bar_e = L == 0 ? bar_e0 : bar_e1;
    const int r16 = rh * 16;                                  // first of the 16 rows whose gates this thread activates
    const int r8 = r16 + (is_b ? 8 : 0);                      // first of the 8 rows whose cell this thread updates
    float c[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) c[r] = 0.f;
    for (int t = 0; t < T; ++t) {
      if (PROF && rec && t >= P0 && t < P0 + PN) tl[t - P0][0] = clock64();
      lt_wait(bar_m, (uint32_t)t & 1u, 1000 * (1 + L) + t);
      if (PROF && rec && t >= P0 && t < P0 + PN) tl[t - P0][1] = clock64();
      tc_fence_after();
      const uint32_t col = L == 0 ? 0u : 64u + (uint32_t)((t & 1) * 64);
      uint32_t v0[16], v1[16];
      tmem_ld16(lane_t + col + (uint32_t)r16, v0);
      tmem_ld16(lane_t + col + 32u + (uint32_t)r16, v1);
      tmem_wait_ld();
      float a0[16], a1[16];
#pragma unroll
      for (int r = 0; r < 16; ++r) {
        a0[r] = sigmoidf_(__uint_as_float(v0[r]) + bias0);
        a1[r] = act_gen(__uint_as_float(v1[r]) + bias1, k1, s1c, o1c);
      }
      if (SAVE) {
        float* s0 = a.stash + stash_index(L, t, T, R, row0 + r16, is_b ? 1 : 0, u);
        float* s1 = a.stash + stash_index(L, t, T, R, row0 + r16, is_b ? 3 : 2, u);
#pragma unroll
        for (int b = 0; b < 2; ++b) {
          st8(s0 + (size_t)b * (5 * 64 * 8), a0[8 * b + 0], a0[8 * b + 1], a0[8 * b + 2], a0[8 * b + 3], a0[8 * b + 4], a0[8 * b + 5],
              a0[8 * b + 6], a0[8 * b + 7]);
          st8(s1 + (size_t)b * (5 * 64 * 8), a1[8 * b + 0], a1[8 * b + 1], a1[8 * b + 2], a1[8 * b + 3], a1[8 * b + 4], a1[8 * b + 5],
              a1[8 * b + 6], a1[8 * b + 7]);
        }
      }
      if (PROF && rec && t >= P0 && t < P0 + PN) tl[t - P0][2] = clock64();
      float hn[8];
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const float p_lo = a0[r] * a1[r], p_hi = a0[8 + r] * a1[8 + r];
        const float x1 = __shfl_xor_sync(0xffffffffu, is_b ? a0[r] : p_hi, 16);   // A lane <- f[r] ; B lane <- (i g)[8 + r]
        const float x2 = __shfl_xor_sync(0xffffffffu, a1[r], 16);                 // A lane <- o[r]
        const float fg = is_b ? a0[8 + r] : x1;
        const float pin = is_b ? x1 : p_lo;
        const float og = is_b ? a1[8 + r] : x2;
        c[r] = fmaf(fg, c[r], pin);
        hn[r] = og * tanhf_(c[r]);
      }
      if (SAVE) {
        st8(a.stash + stash_index(L, t, T, R, row0 + r8, 4, u), c[0], c[1], c[2], c[3], c[4], c[5], c[6], c[7]);
      }
      if (L == 0) {
        uint8_t* dst = sm + LF_H0 + (t & 1) * 2 * LT_OP;
        store_split8(dst, r8 >> 3, u, hn);
      } else {
        if (t >= 1) lt_wait(bar_a, (uint32_t)(t - 1) & 1u, 3000 + t);    // hid2act of step t - 1 is done (implies t - 2: this h1f buffer is free)
        uint8_t* dst = sm + LF_H1;
        float* hf = h1f + (t & 1) * (LT_RB * LF_H1P) + r8 * LF_H1P + u;
#pragma unroll
        for (int r = 0; r < 8; ++r) hf[r * LF_H1P] = hn[r];
        store_split8(dst, r8 >> 3, u, hn);
      }
      if (PROF && rec && t >= P0 && t < P0 + PN) tl[t - P0][3] = clock64();
      tc_fence_before();
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_e);
      if (PROF && rec && t >= P0 && t < P0 + PN) tl[t - P0][4] = clock64();
    }
    if (PROF && rec && (warp == 0 || warp == 8))
      for (int k = 0; k < PN; ++k)
        printf("[fwd prof] warp %2d L%d step %d: top %7lld | mma seen %7lld | acts done %7lld | cell+store done %7lld | arrived %7lld\n", warp, L,
               P0 + k, tl[k][0] - tbase, tl[k][1] - tbase, tl[k][2] - tbase, tl[k][3] - tbase, tl[k][4] - tbase);
  } else if (warp == 16) {
    // ===================== MMA issuer: event loop over the three products of a step =====================
    //   M0(s)  = W0 . [h0_{s-1} ; z_s]        needs E0(s-1), z_s ; and M1a(s-2) issued (it reads the h0 buffer E0(s) rewrites)
    //   M1a(s) = W_ih1 . h0_s  (accumulate 0)  needs E0(s) ; and M1b(s-1) issued => E1(s-2) has read accumulator s & 1
    //   M1b(s) = W_hh1 . h1_{s-1}              needs E1(s-1), after M1a(s)
    // The completed phases of every barrier are counted here (each phase is observed before the next can complete).
    constexpr uint32_t IDESC = idesc_f16(128, LT_RB);
    const uint64_t bh0 = make_desc_nmaj(smem_u32(sm + LF_H0)), bh1 = make_desc_nmaj(smem_u32(sm + LF_H1)), bz = make_desc_nmaj(smem_u32(sm + LF_Z));
    const uint32_t wc = tmem_base + LF_WCOL0;
    // one weight block (TMEM columns `acol` of tile 0, `tstride` columns further for tile 1) against the hi and lo operand tile, nk K = 16 steps
    auto kblock = [&](uint32_t d, uint32_t acol, uint32_t tstride, uint64_t bd, int nk, bool fresh) {
      // consecutive MMAs alternate between the two tiles' accumulators (two independent accumulation chains)
#pragma unroll
      for (int part = 0; part < 2; ++part)
#pragma unroll
        for (int k = 0; k < 4; ++k)
#pragma unroll
          for (int tile = 0; tile < 2; ++tile)
            if (k < nk)
              umma_ts_f16(d + (uint32_t)(tile * 32), acol + (uint32_t)tile * tstride + (uint32_t)(8 * k), bd + (uint64_t)(part * (LT_OP >> 4) + NMAJ_KSTEP * k),
                          IDESC, (fresh && part == 0 && k == 0) ? 0u : 1u);
    };
    int n0 = 0, n1a = 0, n1b = 0, e0_done = 0, e1_done = 0, z_done = 0;
    const long long t_loop = clock64();
    while (n1b < T) {
      if (e0_done < T && mbar_test_wait(bar_e0, (uint32_t)e0_done & 1u)) ++e0_done;
      if (e1_done < T && mbar_test_wait(bar_e1, (uint32_t)e1_done & 1u)) ++e1_done;
      if (z_done < T && mbar_test_wait(bar_z + 8 * (z_done % 3), (uint32_t)(z_done / 3) & 1u)) ++z_done;
      bool progressed = false;
      if (n1b < n1a && e1_done >= n1b) {
        if (PROF && rec && n1b >= P0 && n1b < P0 + PN) tl[n1b - P0][4] = clock64();
        tc_fence_after();
        const uint32_t d1b = tmem_base + 64u + (uint32_t)((n1b & 1) * 64);
        if (elect_one()) {
          kblock(d1b, wc + 80u + 32u, 64u, bh1, 4, false);
          umma_commit(bar_m1);
        }
        __syncwarp();
        if (PROF && rec && n1b >= P0 && n1b < P0 + PN) tl[n1b - P0][5] = clock64();
        ++n1b; progressed = true;
      }
      if (n0 < T && z_done > n0 && e0_done >= n0 && n1a >= n0 - 1) {
        if (PROF && rec && n0 >= P0 && n0 < P0 + PN) tl[n0 - P0][0] = clock64();
        tc_fence_after();
        const uint64_t b_h = bh0 + (uint64_t)(((n0 + 1) & 1) * 2 * (LT_OP >> 4)), b_z = bz + (uint64_t)((n0 % 3) * 2 * (LT_OP >> 4));
        if (elect_one()) {
          kblock(tmem_base, wc, 40u, b_h, 4, true);
          kblock(tmem_base, wc + 32u, 40u, b_z, 1, false);
          umma_commit(bar_m0);
        }
        __syncwarp();
        if (PROF && rec && n0 >= P0 && n0 < P0 + PN) tl[n0 - P0][1] = clock64();
        ++n0; progressed = true;
      }
      if (n1a < T && e0_done > n1a && n1b >= n1a) {
        if (PROF && rec && n1a >= P0 && n1a < P0 + PN) tl[n1a - P0][2] = clock64();
        tc_fence_after();
        const uint32_t d1a = tmem_base + 64u + (uint32_t)((n1a & 1) * 64);
        const uint64_t b_1a = bh0 + (uint64_t)((n1a & 1) * 2 * (LT_OP >> 4));
        if (elect_one()) kblock(d1a, wc + 80u, 64u, b_1a, 4, true);
        __syncwarp();
        if (PROF && rec && n1a >= P0 && n1a < P0 + PN) tl[n1a - P0][3] = clock64();
        ++n1a; progressed = true;
      }
      if (!progressed && clock64() - t_loop > 8000000000ll) {
        if (lane == 0) printf("lstm_tc forward: MMA issuer stuck (block %d, n0 %d n1a %d n1b %d e0 %d e1 %d z %d)\n", (int)blockIdx.x, n0, n1a, n1b, e0_done, e1_done, z_done);
        __trap();
      }
    }
    if (PROF && rec)
      for (int k = 0; k < PN; ++k)
        printf("[fwd prof] mma step %d: M0 %7lld - %7lld | M1a %7lld - %7lld | M1b %7lld - %7lld\n", P0 + k, tl[k][0] - tbase, tl[k][1] - tbase,
               tl[k][2] - tbase, tl[k][3] - tbase, tl[k][4] - tbase, tl[k][5] - tbase);
  } else {
    // ===================== warp 17: z staging, hid2act, unicycle rollout (lane = row) =====================
    const int row = row0 + lane;
    const bool valid = row < R;
    const float hb0 = a.h2a_b[0], hb1 = a.h2a_b[1];
    if (lane == 0) { mbar_arrive(bar_z); mbar_arrive(bar_z + 8); mbar_arrive(bar_z + 16); }      // z_0..z_2 were staged in the prologue
    float4 zn = make_float4(0.f, 0.f, 0.f, 0.f);
    if (valid && 3 < T) zn = reinterpret_cast<const float4*>(a.z)[(size_t)row * T + 3];
    // rollout state (diffuser_helpers.py:573-639), advanced as each action arrives
    const DynParams2& d = a.dyn;
    float px = 0.f, py = 0.f, sp = 0.f, psi = 0.f;
    if (valid) { px = a.curr[(size_t)row * 4 + 0]; py = a.curr[(size_t)row * 4 + 1]; sp = a.curr[(size_t)row * 4 + 2]; psi = a.curr[(size_t)row * 4 + 3]; }
    float vprev = clip2(sp, d.v_lo, d.v_hi);
    for (int s = 1; s <= T; ++s) {
      const int t = s - 1;
      lt_wait(bar_e1, (uint32_t)t & 1u, 20000 + t);
      const float* hf = h1f + (t & 1) * (LT_RB * LF_H1P) + lane * LF_H1P;
      float s0 = hb0, s1 = hb1;
#pragma unroll 16
      for (int k = 0; k < LT_H; ++k) {
        const float hv = hf[k];
        s0 = fmaf(hw[k], hv, s0); s1 = fmaf(hw[LT_H + k], hv, s1);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_a);
      if (s + 2 < T) {
        // stage z_{s+2} over z_{s-1}: E1(s-1) done => M1b(s-1) done => M0(s-1) done (issued earlier, in-order pipe)
        const int slot = (s + 2) % 3;
        uint8_t* zt = sm + LF_Z + slot * 2 * LT_OP;
        store_split(zt, lane, 0, zn.x); store_split(zt, lane, 1, zn.y); store_split(zt, lane, 2, zn.z); store_split(zt, lane, 3, zn.w);
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_z + 8 * slot);
        zn = make_float4(0.f, 0.f, 0.f, 0.f);
        if (valid && s + 3 < T) zn = reinterpret_cast<const float4*>(a.z)[(size_t)row * T + s + 3];
      }
      if (valid) {
        *reinterpret_cast<float2*>(a.act_out + ((size_t)row * T + t) * 2) = make_float2(s0, s1);
        if (a.traj_out) {
          const float a_raw = __fadd_rn(__fmul_rn(s0, d.a_std), d.a_mean);
          const float w_raw = __fadd_rn(__fmul_rn(s1, d.w_std), d.w_mean);
          const float ac = clip2(a_raw, d.acce_lo, d.acce_hi);
          sp = __fadd_rn(sp, __fmul_rn(ac, d.dt));
          const float vnext = clip2(sp, d.v_lo, d.v_hi);
          const float vbar = __fmul_rn(0.5f, __fadd_rn(vprev, vnext));
          const float ve = fabsf(vprev);
          const float yb = fmaxf(fminf(__fmul_rn(d.max_steer, ve), __fdiv_rn(d.max_yawvel, fmaxf(ve, 0.1f))), 0.1f);
          const float w = clip2(w_raw, -yb, yb);
          px = __fadd_rn(px, __fmul_rn(__fmul_rn(vbar, cosf(psi)), d.dt));
          py = __fadd_rn(py, __fmul_rn(__fmul_rn(vbar, sinf(psi)), d.dt));
          psi = __fadd_rn(psi, __fmul_rn(w, d.dt));
          float* o = a.traj_out + ((size_t)row * T + t) * 6;
          *reinterpret_cast<float2*>(o) = make_float2(px, py);
          *reinterpret_cast<float2*>(o + 2) = make_float2(vnext, psi);
          *reinterpret_cast<float2*>(o + 4) = make_float2(a_raw, w_raw);
          vprev = vnext;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 16) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------
// backward (BPTT) on the tensor pipe.  Per step and layer:
//   [dh_rec (64) ; dx (64)]^T [128 x 32 rows] = [W_hh ; W_ih]^T [128 x 256] . dgates^T [256 x 32]
// The M tile's lanes j / j + 16 of a quadrant are (dh_rec[u], dx[u]) of unit u = 16 q + j (layer 1: dx = gradient
// into h0_t; layer 0: dx = dz_t for u < 4).  The gate gradients are the N operand, written by the cell warps as an
// fp16 hi + lo pair after an exact per-row power-of-two scaling (the backward is linear in d(traj) per row), so the
// fp16 range is never the limit and the operand carries ~22 bits relative to the row's largest gradient.
// A cell thread owns one unit and one 8-row stash block: (unit, rows) -> i, f, g, o, c are two 16-byte loads each.
// Layer 0 runs one step behind layer 1 (it needs layer 1's dx of the same time step); layer 1's accumulator is
// double-buffered in TMEM so that layer 0 may still be reading dx while layer 1's next product is written.
// Warp roles (576 threads): warps 0-7 layer-1 cells, 8-15 layer-0 cells (warp & 3 = TMEM lane quadrant,
// (warp >> 2) & 1 = row half), warp 16 MMA issuer, warp 17 idle after the prologue.
// ------------------------------------------------------------------------------------------------
namespace {
constexpr int LB_THREADS = 576;
constexpr int LBK_DG = 0;                               // [layer][hi, lo][gate] x 4 KB (+ 4 KB: the prologue scratch aliases this region)
// 17 operand tiles, or the prologue scratch when that is larger (horizon > 52: 134 KB at T = 104), rounded to 1 KB
__host__ __device__ constexpr int lbk_scr(int T) {
  return (LT_RB * (T * 6 + 4 * (T + 1)) * 4 > 17 * LT_OP) ? ((LT_RB * (T * 6 + 4 * (T + 1)) * 4 + 1023) / 1024) * 1024 : 17 * LT_OP;
}
__host__ __device__ constexpr int lbk_dact(int T) { return LBK_DG + lbk_scr(T); }                 // fp32 [32 rows][T][2], scaled
__host__ __device__ constexpr int lbk_scale(int T) { return lbk_dact(T) + LT_RB * T * 2 * 4; }    // float [32] 1 / scale
__host__ __device__ constexpr int lbk_hw(int T) { return lbk_scale(T) + LT_RB * 4; }             // hid2act weights [2][64]
__host__ __device__ constexpr int lbk_dzs(int T) { return lbk_hw(T) + 2 * LT_H * 4; }            // float [32 rows][4]: dz of one step
__host__ __device__ constexpr int lbk_bars(int T) { return lbk_dzs(T) + LT_RB * 4 * 4; }          // m1[2], m0, e1, e0, dz, dzfree
__host__ __device__ constexpr int lbk_smem(int T) { return lbk_bars(T) + 8 * 8 + 16; }
// prologue scratch (aliases the gate-gradient tiles): act [32][T][2], dtraj [32][T][4], scan scratch [32][4][T+1]
}  // namespace

struct BwdTcArgs {
  const float *z_mean, *act, *curr, *dtraj, *stash;
  const float* dacc;                    // optional [R,T] direct gradient w.r.t. the acceleration command (acc-limit guidance)
  const float* dtraj2;                  // optional second d(traj) part (map-collision kernel on the auxiliary stream), added in the prologue
  const uint8_t* wblob;                 // packed fp16x2 backward weights for TMEM, [256][128]
  const float* h2a_w;
  float *z_out, *grad_out;
  int R, T;
  DynParams2 dyn;
  int optimizer; float lr;
  GuideOpt opt;                         // iteration and Adam moments of a multi-step guided call
  int pf;                               // L2 prefetch distance in steps (0: off)
};

// backward weight blob for TMEM: [256 columns][128 lanes] fp16x2; columns 0..127 layer 1, 128..255 layer 0; column 32 g + c of a
// layer holds gate rows g * 64 + 2 c, + 1 of [W_hh | W_ih]^T for the lane's output (see the kernel comment)
__global__ void lstm_tc_pack_bwd_kernel(uint32_t* __restrict__ out, const float* __restrict__ wih0, const float* __restrict__ whh0,
                                        const float* __restrict__ wih1, const float* __restrict__ whh1) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= LB_WCOLS * 128) return;
  const int m = idx & 127, c = idx >> 7;
  const int layer = c < 128 ? 1 : 0, cc = c & 127;
  const int grow = (cc >> 5) * LT_H + 2 * (cc & 31);
  const int q = m >> 5, l = m & 31, j = l & 15, is_b = l >> 4, u = 16 * q + j;
  float v[2];
  for (int e = 0; e < 2; ++e) {
    const int gr = grow + e;
    if (!is_b) v[e] = (layer == 0 ? whh0 : whh1)[gr * 64 + u];
    else v[e] = layer == 0 ? (u < 4 ? wih0[gr * 4 + u] : 0.f) : wih1[gr * 64 + u];
  }
  const __half2 h = __floats2half2_rn(v[0], v[1]);
  out[idx] = *reinterpret_cast<const uint32_t*>(&h);
}

// 16 columns of the hi accumulator at `taddr` combined with the lo accumulator 32 columns further
__device__ __forceinline__ void tmem_ld16_hilo(uint32_t taddr, float (&o)[16]) {
  uint32_t vh[16], vl[16];
  tmem_ld16(taddr, vh);
  tmem_ld16(taddr + 32, vl);
  tmem_wait_ld();
#pragma unroll
  for (int r = 0; r < 16; ++r) o[r] = fmaf(__uint_as_float(vl[r]), 1.0f / 2048.0f, __uint_as_float(vh[r]));
}

__device__ __forceinline__ void ld8(const float* p, float (&o)[8]) {
  asm volatile("ld.global.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(o[0]), "=f"(o[1]), "=f"(o[2]), "=f"(o[3]), "=f"(o[4]), "=f"(o[5]), "=f"(o[6]), "=f"(o[7]) : "l"(p) : "memory");
}

// MOM: the Adam moments of a multi-step guided call (a.opt.m, a.opt.v) are read / written; the single-iteration instance has no
// moment code at all
template <bool PROF, bool MOM>
__global__ void __launch_bounds__(LB_THREADS, 1) lstm_backward_tc_kernel(const BwdTcArgs a) {
  constexpr int P0 = 20, PN = 4;        // CLD_LSTM_PROF=1: timeline of steps P0 .. P0+PN-1 of CTA 0 (clock64), printed at the end
  long long tl[PN][4];
  const bool rec = PROF && blockIdx.x == 0 && (threadIdx.x & 31) == 0;
  const long long tbase = PROF ? clock64() : 0;
  (void)tl; (void)rec; (void)tbase;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* sm = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int row0 = blockIdx.x * LT_RB, T = a.T, R = a.R;
  const uint32_t bars = smem_u32(sm + lbk_bars(T));
  // bar_m1 alternates between two barriers by step parity: layer 0 (one step behind) waits for MMA_L1(i) while
  // MMA_L1(i + 1) may already complete; a barrier's next completion (step i + 2) needs layer 0's arrival for step i
  const uint32_t bar_m1 = bars, bar_m0 = bars + 16, bar_e1 = bars + 24, bar_e0 = bars + 32, bar_dz = bars + 40, bar_dzfree = bars + 48;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm + lbk_bars(T) + 64);
  float* dzs = reinterpret_cast<float*>(sm + lbk_dzs(T));
  float* dact = reinterpret_cast<float*>(sm + lbk_dact(T));
  float* inv_scale = reinterpret_cast<float*>(sm + lbk_scale(T));
  float* hw = reinterpret_cast<float*>(sm + lbk_hw(T));

  // ---- prologue: d(traj) -> d(scaled action) per row (reverse unicycle scans), per-row scale, weights
  {
    float* act_s = reinterpret_cast<float*>(sm + LBK_DG);            // [32][T][2] (scratch aliases the gate-gradient tiles)
    float* dtr_s = act_s + LT_RB * T * 2;                            // [32][T][4]
    float* scr_s = dtr_s + LT_RB * T * 4;                            // [32][4][T+1]
    const int nrow = min(LT_RB, R - row0);
    for (int i = tid; i < nrow * T * 2 / 4; i += LB_THREADS)
      reinterpret_cast<float4*>(act_s)[i] = reinterpret_cast<const float4*>(a.act + (size_t)row0 * T * 2)[i];
    for (int i = tid; i < nrow * T; i += LB_THREADS) {
      float4 v = reinterpret_cast<const float4*>(a.dtraj + (size_t)row0 * T * 4)[i];
      if (a.dtraj2) {
        const float4 w = reinterpret_cast<const float4*>(a.dtraj2 + (size_t)row0 * T * 4)[i];
        v.x += w.x; v.y += w.y; v.z += w.z; v.w += w.w;
      }
      reinterpret_cast<float4*>(dtr_s)[i] = v;
    }
    if (tid < 2 * LT_H) hw[tid] = a.h2a_w[tid];
    if (tid == 0) {
      mbar_init(bar_m1, 1); mbar_init(bar_m1 + 8, 1); mbar_init(bar_m0, 1); mbar_init(bar_e1, 8); mbar_init(bar_e0, 8);
      mbar_init(bar_dz, 2); mbar_init(bar_dzfree, 1);
      fence_barrier_init();
    }
    if (warp == 16) { tmem_alloc(smem_u32(tmem_slot), 512); tmem_relinquish(); }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp < 16) load_weights_tmem(reinterpret_cast<const uint32_t*>(a.wblob), LB_WCOLS, *tmem_slot + LB_WCOL0, warp & 3, (warp >> 2) & 3, lane);
    if (tid < LT_RB) {
      float* da = dact + tid * T * 2;
      float sc = 1.f;
      if (row0 + tid < R) {
        unicycle_row_backward2(act_s + tid * T * 2, a.curr + (size_t)(row0 + tid) * 4, dtr_s + tid * T * 4, T, a.dyn,
                               scr_s + tid * 4 * (T + 1), da, a.dacc ? a.dacc + (size_t)(row0 + tid) * T : nullptr);
        float m = 0.f;
        for (int i = 0; i < 2 * T; ++i) m = fmaxf(m, fabsf(da[i]));
        if (m > 0.f && m < 3.0e38f) {
          int e;
          frexpf(m, &e);                       // m = f * 2^e, f in [0.5, 1)
          e = max(-100, min(100, e));
          sc = ldexpf(1.f, -e);                // scaled maximum in [0.5, 1)
        }
        for (int i = 0; i < 2 * T; ++i) da[i] *= sc;
      } else {
        for (int i = 0; i < 2 * T; ++i) da[i] = 0.f;
      }
      inv_scale[tid] = 1.f / sc;
    }
    __syncthreads();
    uint4* dg = reinterpret_cast<uint4*>(sm + LBK_DG);
    for (int i = tid; i < 16 * LT_OP / 16; i += LB_THREADS) dg[i] = make_uint4(0u, 0u, 0u, 0u);
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // TMEM columns: layer-1 accumulators [parity][hi 32 | lo 32] at 0..127, layer-0 accumulators [hi | lo] at 128..191,
  // weights (A operand) at 192..447: layer 1 [gate k-block 32 columns] x 4, then layer 0.
  // The lo pass multiplies the residual scaled by 2^11 (so that it is not lost in the fp16 subnormals) into its own
  // accumulator; the cell warps combine  hi + 2^-11 lo.

  if (warp < 16) {
    // ===================== cell-gradient warps =====================
    const int L = warp < 8 ? 1 : 0;
    const int q = warp & 3, rh = (warp >> 2) & 1, j = lane & 15;
    const bool is_b = lane >= 16;
    const int u = 16 * q + j;
    const int rb = rh * 2 + (is_b ? 1 : 0);                 // this thread's 8-row block inside the CTA's 32 rows
    const int rloc = rb * 8;
    const uint32_t lane_t = tmem_base + ((uint32_t)(q * 32) << 16);
    const float hw0 = hw[u], hw1 = hw[LT_H + u];
    const uint32_t bar_e = L ? bar_e1 : bar_e0;
    uint8_t* dgt = sm + LBK_DG + (L ? 0 : 8 * LT_OP);       // [hi, lo][gate] tiles of this layer
    float dcrec[8], cprev[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) dcrec[r] = 0.f;
    for (int i = 0; i <= T; ++i) {
      const int t = T - 1 - i;                                // time step of this iteration (i < T)
      float gi[8], gf[8], gg[8], go[8], cc[8];
      if (a.pf > 0 && (j & 3) == 0 && t - a.pf >= 0) {
        // pull the stash lines of three steps ahead from HBM into L2 (one lane per 128-byte line): the loads below then hit L2
#pragma unroll
        for (int v = 0; v < 5; ++v)
          asm volatile("prefetch.global.L2 [%0];" ::"l"(a.stash + stash_index(L, t - a.pf, T, R, row0 + rloc, v, u)));
      }
      if (i < T) {
        // stash loads first: they do not depend on the MMA and complete while the thread waits below
        ld8(a.stash + stash_index(L, t, T, R, row0 + rloc, 0, u), gi);
        ld8(a.stash + stash_index(L, t, T, R, row0 + rloc, 1, u), gf);
        ld8(a.stash + stash_index(L, t, T, R, row0 + rloc, 2, u), gg);
        ld8(a.stash + stash_index(L, t, T, R, row0 + rloc, 3, u), go);
        ld8(a.stash + stash_index(L, t, T, R, row0 + rloc, 4, u), cc);
        if (t >= 1) ld8(a.stash + stash_index(L, t - 1, T, R, row0 + rloc, 4, u), cprev);
        else {
#pragma unroll
          for (int r = 0; r < 8; ++r) cprev[r] = 0.f;
        }
      }
      if (PROF && rec && i >= P0 && i < P0 + PN) tl[i - P0][0] = clock64();
      float dh[8];
      float v0[16];
#pragma unroll
      for (int r = 0; r < 8; ++r) dh[r] = 0.f;
      if (L == 1) {
        if (i >= T) break;
        if (i >= 1) {
          lt_wait(bar_m1 + 8 * ((i - 1) & 1), (uint32_t)((i - 1) >> 1) & 1u, 31000 + i);
          tc_fence_after();
          float v[16];
          tmem_ld16_hilo(lane_t + (uint32_t)(((i - 1) & 1) * 64 + rh * 16), v);  // A lanes: dh_rec[u] for this row half
#pragma unroll
          for (int r = 0; r < 8; ++r) {
            const float x = __shfl_xor_sync(0xffffffffu, v[8 + r], 16);          // B lane <- A lane's rows 8..15
            dh[r] = is_b ? x : v[r];
          }
        }
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          const float2 da = *reinterpret_cast<const float2*>(dact + ((rloc + r) * T + t) * 2);
          dh[r] = fmaf(hw0, da.x, fmaf(hw1, da.y, dh[r]));
        }
      } else {
        if (i < T) lt_wait(bar_m1 + 8 * (i & 1), (uint32_t)(i >> 1) & 1u, 33000 + i);        // checked first: must be observed before MMA_L1(i + 1) completes
        if (i >= 1) {
          lt_wait(bar_m0, (uint32_t)(i - 1) & 1u, 32000 + i);
          tc_fence_after();
          tmem_ld16_hilo(lane_t + (uint32_t)(128 + rh * 16), v0);               // A: dh_rec0[u] ; B (u < 4): dz of step i - 1
        }
        if (i < T) {
          tc_fence_after();
          float v1[16];
          tmem_ld16_hilo(lane_t + (uint32_t)((i & 1) * 64 + rh * 16), v1);      // B lanes: dx1[u] = d(loss)/d(h0_t)
#pragma unroll
          for (int r = 0; r < 8; ++r) {
            const float rec_lo = i >= 1 ? v0[r] : 0.f, rec_hi = i >= 1 ? v0[8 + r] : 0.f;
            const float send = is_b ? v1[r] : rec_hi;                            // B sends dx rows 0..7 ; A sends dh_rec rows 8..15
            const float x = __shfl_xor_sync(0xffffffffu, send, 16);
            dh[r] = is_b ? (v1[8 + r] + x) : (rec_lo + x);
          }
        }
      }
      if (PROF && rec && i >= P0 && i < P0 + PN) tl[i - P0][1] = clock64();
      if (i < T) {
      // ---- gate gradients of this thread's (unit, 8 rows)
      float dgi[8], dgf[8], dgg[8], dgo[8];
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const float tc = tanhf_(cc[r]);
        const float dc = fmaf(dh[r] * go[r], 1.f - tc * tc, dcrec[r]);
        const float d_i = dc * gg[r] * gi[r] * (1.f - gi[r]);
        const float d_f = dc * cprev[r] * gf[r] * (1.f - gf[r]);
        const float d_g = dc * gi[r] * (1.f - gg[r] * gg[r]);
        const float d_o = dh[r] * tc * go[r] * (1.f - go[r]);
        dcrec[r] = dc * gf[r];
        dgi[r] = d_i; dgf[r] = d_f; dgg[r] = d_g; dgo[r] = d_o;
      }
      // residual scaled by 2^11 so that it is not lost in the fp16 subnormals; one 16-byte store per tile
      store_split8(dgt + 0 * LT_OP, rb, u, dgi, 2048.0f, 4 * LT_OP);
      store_split8(dgt + 1 * LT_OP, rb, u, dgf, 2048.0f, 4 * LT_OP);
      store_split8(dgt + 2 * LT_OP, rb, u, dgg, 2048.0f, 4 * LT_OP);
      store_split8(dgt + 3 * LT_OP, rb, u, dgo, 2048.0f, 4 * LT_OP);
      if (PROF && rec && i >= P0 && i < P0 + PN) tl[i - P0][2] = clock64();
      tc_fence_before();
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_e);
      if (PROF && rec && i >= P0 && i < P0 + PN) tl[i - P0][3] = clock64();
      }
      if (L == 0 && q == 0 && i >= 1) {
        // dz (still scaled) of step index i - 1: staged in shared memory for warp 17, off the critical path (the gate
        // gradients of this step are already published).  One step in flight: wait until warp 17 took the previous one.
        if (i >= 2) lt_wait(bar_dzfree, (uint32_t)(i - 2) & 1u, 34000 + i);
        if (is_b && j < 4) {
#pragma unroll
          for (int r = 0; r < 16; ++r) dzs[(rh * 16 + r) * 4 + j] = v0[r];
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_dz);
      }
    }
    if (PROF && rec && (warp == 0 || warp == 8 || warp == 9 || warp == 13))
      for (int k = 0; k < PN; ++k)
        printf("[bwd prof] warp %2d L%d step %d: top %7lld | waits done %7lld | grads done %7lld | arrived %7lld\n", warp, L, P0 + k,
               tl[k][0] - tbase, tl[k][1] - tbase, tl[k][2] - tbase, tl[k][3] - tbase);
  } else if (warp == 16) {
    // ===================== MMA issuer =====================
    constexpr uint32_t IDESC = idesc_f16(128, LT_RB);
    const uint32_t dg_u = smem_u32(sm + LBK_DG);
    // one product = 2 passes (hi | lo gate gradients, each into its own accumulator) x 4 gate k-blocks x 4 K=16 steps;
    // fully unrolled so that every address is base + immediate
    auto product = [&](const uint32_t a0, const uint64_t b0, const uint32_t d0) {
      // consecutive MMAs alternate between the hi and the lo accumulator (two independent accumulation chains)
#pragma unroll
      for (int g = 0; g < 4; ++g) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
#pragma unroll
          for (int part = 0; part < 2; ++part)
            umma_ts_f16(d0 + (uint32_t)(part * 32), a0 + (uint32_t)(g * 32 + 8 * k), b0 + (uint64_t)((part * 4 + g) * (LT_OP >> 4) + NMAJ_KSTEP * k), IDESC,
                        (g | k) ? 1u : 0u);
        }
      }
    };
    const uint32_t a_l1 = tmem_base + LB_WCOL0, a_l0 = tmem_base + LB_WCOL0 + 128u;
    const uint64_t b_l1 = make_desc_nmaj(dg_u), b_l0 = make_desc_nmaj(dg_u + 8u * LT_OP);
    // event loop: issue whichever layer's product has its operand ready, so that neither recurrence chain waits
    // behind the other's barrier.  n1 / n0 = products issued so far.  M1(n1) overwrites accumulator n1 & 1, which
    // layer 0 reads in step n1 - 2: that step is complete once M0(n1 - 2) has been issued (n0 >= n1 - 1).
    int n1 = 0, n0 = 0;
    const long long t_loop = clock64();
    while (n0 < T) {
      bool progressed = false;
      if (n1 < T && (n1 < 2 || n0 >= n1 - 1) && mbar_test_wait(bar_e1, (uint32_t)n1 & 1u)) {
        if (PROF && rec && n1 >= P0 && n1 < P0 + PN) tl[n1 - P0][0] = clock64();
        tc_fence_after();
        const uint32_t d1 = tmem_base + (uint32_t)((n1 & 1) * 64), bm = bar_m1 + 8 * (n1 & 1);
        if (elect_one()) { product(a_l1, b_l1, d1); umma_commit(bm); }
        __syncwarp();
        if (PROF && rec && n1 >= P0 && n1 < P0 + PN) tl[n1 - P0][1] = clock64();
        ++n1;
        progressed = true;
      }
      if (n0 < n1 && mbar_test_wait(bar_e0, (uint32_t)n0 & 1u)) {
        if (PROF && rec && n0 + 1 >= P0 && n0 + 1 < P0 + PN) tl[n0 + 1 - P0][2] = clock64();
        tc_fence_after();
        if (elect_one()) { product(a_l0, b_l0, tmem_base + 128u); umma_commit(bar_m0); }
        __syncwarp();
        if (PROF && rec && n0 + 1 >= P0 && n0 + 1 < P0 + PN) tl[n0 + 1 - P0][3] = clock64();
        ++n0;
        progressed = true;
      }
      if (!progressed && clock64() - t_loop > 8000000000ll) {
        if (lane == 0) printf("lstm_tc backward: MMA issuer stuck (block %d, n1 %d, n0 %d)\n", (int)blockIdx.x, n1, n0);
        __trap();
      }
    }
    if (PROF && rec)
      for (int k = 0; k < PN; ++k)
        printf("[bwd prof] mma s %d: e1 ok %7lld | L1 issued %7lld | e0 ok %7lld | L0 issued %7lld\n", P0 + k, tl[k][0] - tbase,
               tl[k][1] - tbase, tl[k][2] - tbase, tl[k][3] - tbase);
  }
  else {
    // ===================== warp 17: dz -> optimizer step on z (guidance_loss.py:2250-2278), lane = row =====================
    const int row = row0 + lane;
    const bool valid = row < R;
    const float is = inv_scale[lane], lr = a.lr;
    const bool adam = a.optimizer == CLD_OPT_ADAM;
    // Adam moments of a multi-step call: iteration 1 writes them, later iterations read them back (the moments see the
    // unscaled gradient, as grad_out does)
    const bool mom = MOM && adam, mom_in = mom && a.opt.iter > 1;
    auto upd = [&](float z, float g) {
      float m, vv;
      if (adam) return adam_first_step(z, g, lr, m, vv);
      return z - lr * g;
    };
    auto upd_m = [&](float z, float g, float& m, float& vv) {
      if (mom_in) return adam_next_step(z, g, a.opt.step_size, a.opt.bc2_sqrt, m, vv);
      return adam_first_step(z, g, lr, m, vv);
    };
    const float4* zin = reinterpret_cast<const float4*>(a.z_mean);
    float4* mp = reinterpret_cast<float4*>(a.opt.m);
    float4* vp = reinterpret_cast<float4*>(a.opt.v);
    float4 z = make_float4(0.f, 0.f, 0.f, 0.f), m4 = z, v4 = z;
    if (valid) z = zin[(size_t)row * T + (T - 1)];
    if (valid && mom_in) { m4 = mp[(size_t)row * T + (T - 1)]; v4 = vp[(size_t)row * T + (T - 1)]; }
    for (int i = 1; i <= T; ++i) {
      const int tz = T - i;
      lt_wait(bar_dz, (uint32_t)(i - 1) & 1u, 50000 + i);
      float4 g = reinterpret_cast<const float4*>(dzs)[lane];
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_dzfree);
      g.x *= is; g.y *= is; g.z *= is; g.w *= is;
      const float4 zc = z;
      float4 mn = m4, vn = v4;
      if (valid && tz >= 1) {
        z = zin[(size_t)row * T + tz - 1];                  // next step's z (and moments), in flight during this step
        if (mom_in) { m4 = mp[(size_t)row * T + tz - 1]; v4 = vp[(size_t)row * T + tz - 1]; }
      }
      if (valid) {
        const size_t o = (size_t)row * T + tz;
        if (!mom) {
          reinterpret_cast<float4*>(a.z_out)[o] = make_float4(upd(zc.x, g.x), upd(zc.y, g.y), upd(zc.z, g.z), upd(zc.w, g.w));
        } else {
          float4 zn;
          zn.x = upd_m(zc.x, g.x, mn.x, vn.x); zn.y = upd_m(zc.y, g.y, mn.y, vn.y);
          zn.z = upd_m(zc.z, g.z, mn.z, vn.z); zn.w = upd_m(zc.w, g.w, mn.w, vn.w);
          reinterpret_cast<float4*>(a.z_out)[o] = zn;
          mp[o] = mn; vp[o] = vn;
        }
        if (a.grad_out) reinterpret_cast<float4*>(a.grad_out)[o] = g;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 16) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static int lf_smem_req() { return LF_SMEM + 1024 > LT_MIN_SMEM ? LF_SMEM + 1024 : LT_MIN_SMEM; }
static int lb_smem_req(int T) { return lbk_smem(T) + 1024 > LT_MIN_SMEM ? lbk_smem(T) + 1024 : LT_MIN_SMEM; }

struct LstmTcState {
  uint8_t* wfwd = nullptr;
  uint8_t* wbwd = nullptr;
};

static int lstm_tc_prepare(CldHandle* h, cudaStream_t s) {
  if (h->lstm_tc) return 0;
  DecoderW& w = h->dec;
  LstmTcState* st = new LstmTcState();
  CLD_CUDA_OK(h, cudaMalloc((void**)&st->wfwd, (size_t)LF_WCOLS * 128 * 4));
  h->allocs.push_back(st->wfwd);
  lstm_tc_pack_fwd_kernel<<<(LF_WCOLS * 128 + 255) / 256, 256, 0, s>>>(reinterpret_cast<uint32_t*>(st->wfwd), w.wih0_raw, w.whh0_raw, w.wih1_raw, w.whh1_raw);
  CLD_LAUNCH_OK(h, "lstm_tc_pack_fwd_kernel");
  CLD_CUDA_OK(h, cudaFuncSetAttribute(lstm_decode_tc_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, lf_smem_req()));
  CLD_CUDA_OK(h, cudaFuncSetAttribute(lstm_decode_tc_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, lf_smem_req()));
  CLD_CUDA_OK(h, cudaFuncSetAttribute(lstm_decode_tc_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, lf_smem_req()));
  CLD_CUDA_OK(h, cudaMalloc((void**)&st->wbwd, (size_t)LB_WCOLS * 128 * 4));
  h->allocs.push_back(st->wbwd);
  lstm_tc_pack_bwd_kernel<<<(LB_WCOLS * 128 + 255) / 256, 256, 0, s>>>(reinterpret_cast<uint32_t*>(st->wbwd), w.wih0_raw, w.whh0_raw, w.wih1_raw, w.whh1_raw);
  CLD_LAUNCH_OK(h, "lstm_tc_pack_bwd_kernel");
  if (lbk_smem(h->cfg.horizon) + 1024 > 232448) return fail(h, CLD_ERR_UNSUPPORTED, "horizon too long for the tensor-core LSTM backward");
  CLD_CUDA_OK(h, cudaFuncSetAttribute(lstm_backward_tc_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, lb_smem_req(h->cfg.horizon)));
  CLD_CUDA_OK(h, cudaFuncSetAttribute(lstm_backward_tc_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, lb_smem_req(h->cfg.horizon)));
  CLD_CUDA_OK(h, cudaFuncSetAttribute(lstm_backward_tc_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, lb_smem_req(h->cfg.horizon)));
  h->lstm_tc = st;
  return 0;
}

void lstm_tc_destroy(CldHandle* h) {
  if (h->lstm_tc) { delete reinterpret_cast<LstmTcState*>(h->lstm_tc); h->lstm_tc = nullptr; }
}

int decode_rollout_h0_tc(CldHandle* h, const float* z, const float* h0, const float* curr, float* act_out, float* traj_out,
                         bool save, int R, cudaStream_t s) {
  DecoderW& w = h->dec;
  if (!w.loaded) return fail(h, CLD_ERR_STATE, "decoder weights not loaded");
  if (h->cfg.hidden != LT_H || h->cfg.latent_dim != 4) return fail(h, CLD_ERR_UNSUPPORTED, "decoder kernel is specialised for hidden=64, latent=4");
  int rc;
  if ((rc = lstm_tc_prepare(h, s))) return rc;
  const LstmTcState* st = reinterpret_cast<const LstmTcState*>(h->lstm_tc);
  LstmTcArgs a;
  a.z = z; a.h0 = h0; a.curr = curr; a.wblob = st->wfwd; a.b0 = w.b0; a.b1 = w.b1;
  a.h2a_w = w.h2a_w; a.h2a_b = w.h2a_b; a.act_out = act_out; a.traj_out = traj_out; a.stash = save ? h->stash : nullptr;
  a.R = R; a.T = h->cfg.horizon; a.dyn = make_dyn2(h->cfg);
  const int grid = (R + LT_RB - 1) / LT_RB;
  if (save) lstm_decode_tc_kernel<true, false><<<grid, LT_THREADS, lf_smem_req(), s>>>(a);
  else if (h->env_lstm_prof) lstm_decode_tc_kernel<false, true><<<grid, LT_THREADS, lf_smem_req(), s>>>(a);
  else lstm_decode_tc_kernel<false, false><<<grid, LT_THREADS, lf_smem_req(), s>>>(a);
  CLD_LAUNCH_OK(h, "lstm_decode_tc_kernel");
  return 0;
}


int decode_backward_update_tc(CldHandle* h, const float* z_mean, const float* act, const float* curr, const float* dtraj,
                              const float* dtraj2, const float* dacc, const CldGuidanceConfig* g, const GuideOpt& opt, float* z_out,
                              float* grad_out, int R, cudaStream_t s) {
  int rc;
  if ((rc = lstm_tc_prepare(h, s))) return rc;
  const LstmTcState* st = reinterpret_cast<const LstmTcState*>(h->lstm_tc);
  BwdTcArgs a;
  a.z_mean = z_mean; a.act = act; a.curr = curr; a.dtraj = dtraj; a.dtraj2 = dtraj2; a.dacc = dacc; a.stash = h->stash; a.wblob = st->wbwd;
  a.h2a_w = h->dec.h2a_w; a.z_out = z_out; a.grad_out = grad_out; a.R = R; a.T = h->cfg.horizon; a.dyn = make_dyn2(h->cfg);
  a.optimizer = g->optimizer; a.lr = g->lr; a.opt = opt;
  a.pf = h->env_lstm_pf;
  const int grid = (R + LT_RB - 1) / LT_RB;
  if (opt.m) lstm_backward_tc_kernel<false, true><<<grid, LB_THREADS, lb_smem_req(a.T), s>>>(a);
  else if (h->env_lstm_prof) lstm_backward_tc_kernel<true, false><<<grid, LB_THREADS, lb_smem_req(a.T), s>>>(a);
  else lstm_backward_tc_kernel<false, false><<<grid, LB_THREADS, lb_smem_req(a.T), s>>>(a);
  CLD_LAUNCH_OK(h, "lstm_backward_tc_kernel");
  return 0;
}

}  // namespace cld
