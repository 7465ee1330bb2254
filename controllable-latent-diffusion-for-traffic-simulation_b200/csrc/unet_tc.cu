// bf16 tensor-core denoiser: TemporalMapUnet.forward (reference src/tbsim/models/temporal.py:122-180) as ONE
// persistent sm_100a kernel.  A CTA owns a group of 8 batch rows and carries them through all 35
// convolutions with the activations resident in shared memory (bf16, channels-last, 128B-swizzled) and the
// accumulators in tensor memory; the 8.7 MB bf16 weight set is streamed from L2 through a 16 x 4 KB ring by the
// bulk-copy (TMA) unit.  Layout trick: GEMM row m = time_slot * 8 + batch_row, so a convolution tap is a shift
// by whole 1024-byte swizzle atoms of the SAME shared-memory tile (5 taps = 5 UMMA descriptors, no im2col),
// stride-2 convolutions are the same descriptor with SBO = 2048, the transposed convolution is two output
// phases.  GroupNorm statistics are CTA-local because a CTA holds whole rows; GroupNorm + Mish + time/cond bias
// + residual are fused into the TMEM -> register -> shared-memory epilogue that writes the next layer's A operand.
//
// Pipelining inside a row group: the output channels of the wide layers (N >= 128) are computed as two halves
// (GroupNorm groups 0-3 | 4-7).  The epilogue of half 0 runs while the tensor pipe computes half 1, and the next
// layer's MMAs start on the input channels produced by half 0 while the epilogue of half 1 is still running
// (act[h] / acc[h] mbarrier pairs; the k-blocks of an op are ordered G0 | G1 | G2, see TcOp).
//
// Warp roles (576 threads): warps 0..15 epilogue, warp 16 weight producer, warp 17 MMA issuer (one elected thread)
// (4 warps per TMEM lane quadrant; one GroupNorm group per warp per half, 32 accumulator values per thread held
// in registers between the statistics pass and the normalise pass).
#include <stdlib.h>

#include <type_traits>
#include <vector>

#include <cuda.h>

#include "tc_common.cuh"
#include "unet_tc.cuh"

namespace cld {
using namespace tc;

constexpr int TC_G = 8;
constexpr int TC_UNIT = 4096;
constexpr int TC_UNITS = 16;
// weight ring (64 KB): every k-block takes one slot.  Single-CTA kernel: 4 slots of 16 KB (<= 128 weight rows x 128 B);
// CTA-pair kernel: each CTA stages HALF of the rows of a k-block, 8 slots of 8 KB -> twice as many k-blocks in flight for the
// same L2 -> SM bytes (the level-2 layers are bound by the latency of this stream, tools/umma_bench.cu)
// A slot carries a GROUP of consecutive k-blocks of one op (as many as fit): the issuer pays one full-barrier wait and one
// ring-release commit per group, not per k-block -- with 4 MMAs per barrier round trip the single issuing thread, not the
// tensor pipe, set the pace of the N = 256 layers (measured ~550 cycles per k-block for 256 cycles of math).
template <bool PAIR> struct Ring { static constexpr int SLOT = 16384, SLOTS = 4; };
static_assert(Ring<false>::SLOT * Ring<false>::SLOTS == TC_UNIT * TC_UNITS && Ring<true>::SLOT * Ring<true>::SLOTS == TC_UNIT * TC_UNITS, "ring size");
constexpr int TC_EW = 16;                       // epilogue warps
constexpr int TC_ETHREADS = TC_EW * 32;
constexpr int TC_THREADS = 64 + TC_ETHREADS;
constexpr int TC_ARENA = 136 * 1024;   // split-time mode at level 2: 2 regions x 4 panels x (13 + 4) slots
constexpr int TB_LD = 260;            // padded row stride of the time-bias tile (bank-conflict free float4 reads)
constexpr int PAR_ROWS = 5;           // conv bias, GN gamma, GN beta, residual-conv bias, time vector
constexpr int TC_MAX_OPS = 32;
constexpr int TC_MAX_KBS = 768;
constexpr int TC_RES_COL = 256;       // TMEM: accumulators in columns [0,256), residual 1x1 conv in [256,512)

enum { EPI_GN_TB = 0, EPI_GN_RES_ACC = 1, EPI_GN_RES_ID = 2, EPI_BIAS = 3, EPI_UP = 4, EPI_GN = 5, EPI_OUT = 6 };
enum { F_SPLIT_K = 1, F_COMMIT_SPLIT = 2 };

// One fused op = convolution(s) into TMEM + an epilogue.  k-blocks are issued in three groups:
//   wait act[0] (and act[1] unless F_SPLIT_K) | G0 | wait act[1] | G1 | commit acc[0] if F_COMMIT_SPLIT | G2 |
//   commit acc[0] unless F_COMMIT_SPLIT | commit acc[1]
struct TcOp {
  int n_tiles, tile_slot0[4], tile_lo[4], tile_hi[4];
  int sbo, slot_stride;
  int kb_first, n_g0, n_g1, n_g2, flags;
  int epi, n, cout, cpg, t_out, n_vt;
  int dst_off, dst_pitch;
  int par_off, tb_off;
  int zero_pitch, zero_npanels, zero_offB;     // zero_pitch == 0: no halo zeroing
  int save_skip;                               // -1 or byte offset inside the CTA's skip buffer
  int load_skip, load_off, load_pitch, load_npanels, load_T;   // load_skip: -1 or byte offset in the skip buffer
  int dbg_stage;
  int pad_[4];
};
static_assert(sizeof(TcOp) % 16 == 0, "TcOp is copied as uint4");

// host-side k-block record; the device gets it packed in 32 bits:
//   [0,8) A start in 1 KB slots (panel base + tap shift) | [8,14) TMEM column / 8 | [14,20) MMA N / 8 |
//   [20,23) number of K=16 steps | [23] first (overwrite accumulator) | [24,26) log2(ring units) |
//   [26] first k-block of its ring slot (wait for the slot) | [27] last k-block of its ring slot (release the slot)
struct TcKb { int a_base, shift, w_off, acc_col, n, nk16, first, units, slot_first, slot_last; };

// shared-memory layout (byte offsets from the 1024-aligned base)
constexpr int SM_RING = TC_ARENA;
constexpr int SM_PAR = SM_RING + TC_UNITS * TC_UNIT;          // float [2][PAR_ROWS][256]
constexpr int SM_TB = SM_PAR + 2 * PAR_ROWS * 256 * 4;        // float [8][TB_LD]
constexpr int SM_ST = SM_TB + TC_G * TB_LD * 4;               // float2 [2][4 cq][4 quadrants][8 rows]
constexpr int SM_KBS = SM_ST + 2 * 4 * 4 * 8 * 8;             // uint32 [TC_MAX_KBS] (the producer's k-block records)
constexpr int SM_BARS = SM_KBS + TC_MAX_KBS * 4;              // full[16], empty[16], act[2], acc[2]
constexpr int SM_GLOB = SM_BARS + 40 * 8;                     // TcShared
constexpr int TC_SMEM = SM_GLOB + 32;
struct TcShared { uint32_t tmem_base, pad; uint8_t* skip_cta; };
static_assert(TC_SMEM <= 232448, "shared memory budget");

// What the MMA issuer reads, passed BY VALUE as a kernel parameter: it lives in the constant bank, so the (warp-uniform) loop
// counters index it with uniform loads and the whole descriptor arithmetic stays on the uniform datapath.  Read from shared
// memory the same values arrive in per-lane registers and every operand of every tcgen05.mma costs an R2UR: ~90 instructions per
// k-block, ~450 cycles of a single warp's dependent issue for 256 cycles of math in the N = 256 layers.
struct TcIssueOp { int n_g0, n_g1, n_g2, flags, n, nt, sbo, ts[4]; };     // ts: A start of m-tile i in 16-byte units (tile_slot0 * slot_stride * 64)
// one record per k-block -- or per PAIR of consecutive k-blocks of a single-m-tile op (KB_DUAL: the issuer's loop overhead per
// iteration, ~300 cycles of barrier / constant-load / elect latency, is then paid once per 8 MMAs instead of once per 4):
// x = A start (16-byte units from the arena base), y = A start of the second k-block, z = instruction descriptor,
// w = [0] four K=16 steps (else one) | [1] accumulate | [2] first record of its ring slot | [3] last one | [4] dual |
//     [5,14) TMEM column of the accumulator | [16,32) bytes / 16 this CTA stages per k-block
enum { KB_K4 = 1, KB_ACC = 2, KB_SLOT_FIRST = 4, KB_SLOT_LAST = 8, KB_DUAL = 16 };
// `ops`: the full op records for the epilogue warps (uniform loads instead of a chain of shared-memory loads per op and half)
struct TcIssueTab { int n_ops, n_kbs; TcIssueOp op[TC_MAX_OPS]; uint4 kb[TC_MAX_KBS]; TcOp ops[TC_MAX_OPS]; };
static_assert(sizeof(TcIssueTab) + 4 * 128 + 256 < 32000, "kernel parameters");

struct TcParams {
  const TcOp* ops; int n_ops; const uint32_t* kbs; int n_kbs;
  const uint8_t* wblob; size_t wcopy_stride; int wcopies; int w_rows_per_copy; const float* par; const float* tbias; const float* tvec; int tb_stride;
  const float* x; float* eps; int R, T, n_groups;
  // split-time mode (horizon 2 * T, e.g. 104): a CTA carries 4 rows; GEMM lane b = half * 4 + row holds time [half * T, (half + 1) * T)
  // of row b & 3, so the arena / tensor-memory budget is the one of T.  The two halves of a row meet at the inner edges: every
  // panel has its own leading and trailing halo (pitch T' + 4 slots), the inner ones carry copies of the partner lane's edge slots
  // (written by whoever writes the data), the outer ones are zero; GroupNorm statistics are summed over both lanes of a row.
  int tsplit;
  uint8_t* skipbuf; int skip_stride;
  int zero0_pitch, zero0_npanels, zero0_offB;
  int dbg_stage; float* dbg_out;
  long long* prof;   // optional [gridDim][8] cycle counters (CLD_TC_PROF=1): see tc_launch
};

struct TcState {
  std::vector<TcOp> ops;
  std::vector<TcKb> kbs;
  TcOp* d_ops = nullptr; uint32_t* d_kbs = nullptr;
  uint8_t* wblob = nullptr; size_t wblob_bytes = 0; int wcopies = 1;
  TcIssueTab* itab = nullptr;          // host copy of the issuer's table
  bool tsplit = false; int t_eff = 0;   // split-time mode (horizon > 56): lanes of t_eff = horizon / 2 steps
  int zero0_pitch = 0, zero0_offB = 0;
  bool pair = false;                    // CTA-pair kernel (cluster of 2, tcgen05 cta_group::2); CLD_TC_PAIR=0 selects the single-CTA kernel
  CUtensorMap tm8, tm16, tm32, tm64;    // the weight blob as a 2-D tensor {64 bf16, rows}; boxes of 8 / 16 / 32 / 64 rows = half a k-block
  float* par = nullptr; size_t par_floats = 0;
  float* zeros = nullptr;
  long long* prof = nullptr;
  uint8_t* skipbuf = nullptr; int skip_stride = 0; int grid = 0;
  bool ready = false;
};

// ------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float mish_fast(float x) {
  // x * tanh(softplus(x)) = x * n / (n + 2) = x * (1 - 2 / (n + 2)),  n = e^x (e^x + 2); inf-safe (1/inf = 0)
  float e = __expf(x);
  float d = fmaf(e, e + 2.f, 2.f);
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(d));
  return x * fmaf(r, -2.f, 1.f);
}
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float2 unpack_bf16(uint32_t u) {
  __nv_bfloat162 v = *reinterpret_cast<__nv_bfloat162*>(&u);
  return __bfloat1622float2(v);
}
__device__ __forceinline__ void epi_bar() { named_bar(1, TC_ETHREADS); }


// batch row of GEMM lane b of group g; split-time mode: 4 rows per group, lane b = half * 4 + row
__device__ __forceinline__ int row_of(int g, int b, int tsplit) { return tsplit ? g * 4 + (b & 3) : g * TC_G + b; }

// split-time mode: outer halos = leading halo (slots 0, 1 of the panel) of the half-0 lanes (rows 0..3 of the slot) and trailing halo
// (slots T' + 2, T' + 3) of the half-1 lanes (rows 4..7); 512 bytes each, both regions, every panel
__device__ __forceinline__ void zero_halos_split(uint8_t* arena, int offB, int pitch, int npanels, int etid) {
  const int per_panel = 2 * 2 * 32;                 // {leading, trailing} x 2 slots x 32 uint4 (4 rows x 128 B)
  for (int i = etid; i < 2 * npanels * per_panel; i += TC_ETHREADS) {
    const int w = i & 31, sl = (i >> 5) & 1, tr = (i >> 6) & 1, pp = i >> 7;
    const int reg = pp / npanels, p = pp - reg * npanels;
    uint8_t* base = arena + (reg ? offB : 0) + p * pitch;
    uint4* dst = reinterpret_cast<uint4*>(base + (tr ? (pitch - 2048 + sl * 1024 + 512) : sl * 1024)) + w;
    *dst = make_uint4(0u, 0u, 0u, 0u);
  }
}

__device__ __forceinline__ void zero_halos(uint8_t* arena, int offB, int pitch, int npanels, int etid) {
  // per region: leading 2 slots of every panel + 2 tail slots after the last panel = (npanels+1) blocks of 2 KB
  const int blocks = 2 * (npanels + 1);
  for (int i = etid; i < blocks * 128; i += TC_ETHREADS) {
    int blk = i >> 7, w = i & 127;
    int reg = blk / (npanels + 1), p = blk % (npanels + 1);
    uint4* dst = reinterpret_cast<uint4*>(arena + (reg ? offB : 0) + p * pitch) + w;
    *dst = make_uint4(0u, 0u, 0u, 0u);
  }
}

__device__ __forceinline__ void tmem_ldn(uint32_t taddr, uint32_t (&r)[8]) { tmem_ld8(taddr, r); }
__device__ __forceinline__ void tmem_ldn(uint32_t taddr, uint32_t (&r)[16]) { tmem_ld16(taddr, r); }
__device__ __forceinline__ void tmem_ldn(uint32_t taddr, uint32_t (&r)[32]) { tmem_ld32(taddr, r); }

// tcgen05.mma with the 64-bit descriptors given as (low, high) words: the start-address field lives in the low word and never
// carries, so a tap / K-step / tile offset is ONE 32-bit add instead of an add-with-carry pair
template <bool PAIR>
__device__ __forceinline__ void umma_lohi(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc, uint32_t accumulate) {
  if (PAIR)
    asm volatile("{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tmov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\tsetp.ne.b32 p, %6, 0;\n\t"
                 "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %5, p;\n\t}"
                 ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate) : "memory");
  else
    asm volatile("{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tmov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\tsetp.ne.b32 p, %6, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}"
                 ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate) : "memory");
}

struct EpiCtx {
  uint8_t* arena; const float* par; const float* tb_s; float2* st; uint32_t lane_addr;
  int q, cq, lane, etid, g, tsplit;
  uint8_t* skip_cta; float* dbg_out; int dbg_stage; int R;
  long long* tl;   // profiling build only: per-item phase timestamps
};

// split-time mode: an edge slot of lane b is also the inner halo of its partner lane (the other half of the same row): the first two
// slots of a half-1 lane are the trailing halo (slots T', T' + 1) of lane b - 4, the last two of a half-0 lane the leading halo
// (slots -2, -1) of lane b + 4.  `panel` = start of the panel (its slot -2).
__device__ __forceinline__ void store_inner_halo(uint8_t* panel, int t_out, int slot, int b, int c, const uint4& pk) {
  int bp, hs;
  if (b >= 4 && slot < 2) { bp = b - 4; hs = t_out + 2 + slot; }
  else if (b < 4 && slot >= t_out - 2) { bp = b + 4; hs = slot - (t_out - 2); }
  else return;
  *reinterpret_cast<uint4*>(panel + hs * 1024 + bp * 128 + ((((c >> 3) & 7) ^ bp) << 4)) = pk;
}

// store 8 consecutive channels of one (slot, batch row) as bf16: next layer's A operand (+ skip buffer, + debug tap)
__device__ __forceinline__ void store_chunk(const TcOp* o, const EpiCtx& cx, const float (&y)[8], int c, int slot, int b, bool valid) {
  if (!valid || c >= o->cout) return;
  uint4 pk = make_uint4(pack_bf16(y[0], y[1]), pack_bf16(y[2], y[3]), pack_bf16(y[4], y[5]), pack_bf16(y[6], y[7]));
  const int sw = ((((c >> 3) & 7) ^ b) << 4);
  *reinterpret_cast<uint4*>(cx.arena + o->dst_off + (slot + 2) * 1024 + b * 128 + (c >> 6) * o->dst_pitch + sw) = pk;
  if (cx.tsplit) store_inner_halo(cx.arena + o->dst_off + (c >> 6) * o->dst_pitch, o->t_out, slot, b, c, pk);
  if (o->save_skip >= 0)
    *reinterpret_cast<uint4*>(cx.skip_cta + o->save_skip + ((size_t)(c >> 6) * o->t_out + slot) * 1024 + b * 128 + sw) = pk;
}

// debug tap: copy the finished output of op `o` (bf16, in the arena) to the fp32 tap buffer [R][t_out][cout]
__device__ __forceinline__ void dump_stage(const TcOp* o, const EpiCtx& cx) {
  const int chunks = o->cout >> 3, total = o->t_out * TC_G * chunks;
  for (int i = cx.etid; i < total; i += TC_ETHREADS) {
    const int ch = i % chunks, b = (i / chunks) & 7, slot = i / (chunks * 8), c = ch * 8;
    const int row = row_of(cx.g, b, cx.tsplit);
    if (row >= cx.R) continue;
    const uint4 pk = *reinterpret_cast<const uint4*>(cx.arena + o->dst_off + (slot + 2) * 1024 + b * 128 + (c >> 6) * o->dst_pitch +
                                                     ((((c >> 3) & 7) ^ b) << 4));
    float* dp = cx.tsplit ? cx.dbg_out + ((size_t)row * 2 * o->t_out + (b >> 2) * o->t_out + slot) * o->cout + c
                          : cx.dbg_out + ((size_t)row * o->t_out + slot) * o->cout + c;
    float2 f0 = unpack_bf16(pk.x), f1 = unpack_bf16(pk.y), f2 = unpack_bf16(pk.z), f3 = unpack_bf16(pk.w);
    dp[0] = f0.x; dp[1] = f0.y; dp[2] = f1.x; dp[3] = f1.y; dp[4] = f2.x; dp[5] = f2.y; dp[6] = f3.x; dp[7] = f3.y;
  }
}

// GroupNorm + Mish (+ time bias | + residual) for ONE GroupNorm group (CPG channels) of one half of the op,
// over the warp's 32 GEMM rows x NVT m-tiles.  NVT * CPG values per thread stay in registers between the passes;
// both passes walk them in 8-channel chunks with compiler barriers in between to keep the live set small.
#ifdef TC_NO_FENCE
#define TC_SCHED_FENCE()
#else
#define TC_SCHED_FENCE() asm volatile("" ::: "memory")
#endif
__device__ __forceinline__ EpiCtx make_epi_ctx(uint8_t* smem, const float* par) {
  EpiCtx cx;
  const int tid = threadIdx.x, warp = tid >> 5;
  cx.etid = tid; cx.q = warp & 3; cx.cq = warp >> 2; cx.lane = tid & 31;
  cx.arena = smem; cx.par = par;
  cx.tb_s = reinterpret_cast<const float*>(smem + SM_TB); cx.st = reinterpret_cast<float2*>(smem + SM_ST);
  const TcShared* gs = reinterpret_cast<const TcShared*>(smem + SM_GLOB);
  cx.lane_addr = gs->tmem_base + ((uint32_t)(cx.q * 32) << 16);
  cx.skip_cta = gs->skip_cta;
  cx.g = 0; cx.dbg_out = nullptr; cx.dbg_stage = -1; cx.R = 0; cx.tl = nullptr; cx.tsplit = 0;
  return cx;
}

// packed fp32 pairs (FADD2 / FMUL2 / FFMA2): half the issue slots of the scalar forms
__device__ __forceinline__ uint64_t pk2(float a, float b) { uint64_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ uint64_t pk2u(uint32_t a, uint32_t b) { uint64_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(a), "r"(b)); return r; }
__device__ __forceinline__ void upk2(uint64_t p, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(p)); }
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) { uint64_t r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ uint64_t mul2(uint64_t a, uint64_t b) { uint64_t r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) { uint64_t r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ float ex2_ftz(float x) { float r; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float rcp_ftz(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ uint32_t pack_bf16_2(uint64_t p) { float a, b; upk2(p, a, b); return pack_bf16(a, b); }

// Mish on a packed pair whose input is ALREADY scaled by log2(e):  t' = log2e * x  ->  x * tanh(softplus(x))
//   e = 2^t' = exp(x); n = e (e + 2); tanh(softplus(x)) = n / (n + 2) = 1 - 2 / (n + 2); x = ln2 * t'
__device__ __forceinline__ uint64_t mish2_log2(uint64_t t) {
  float tx, ty;
  upk2(t, tx, ty);
  const uint64_t e = pk2(ex2_ftz(tx), ex2_ftz(ty));
  const uint64_t two = pk2(2.f, 2.f);
  const uint64_t d = fma2(e, add2(e, two), two);
  float dx, dy;
  upk2(d, dx, dy);
  const uint64_t w = fma2(pk2(rcp_ftz(dx), rcp_ftz(dy)), pk2(-1.3862943611198906f, -1.3862943611198906f),
                          pk2(0.6931471805599453f, 0.6931471805599453f));
  return mul2(t, w);
}

// GroupNorm + Mish (+ time bias | + residual) for ONE GroupNorm group (cpg channels) of one half of the op, over the
// warp's 32 GEMM rows.  The thread's values are `nch` chunks of 8 channels held in registers between the statistics
// pass and the normalise pass; chunk k belongs to m-tile k / cpt and covers channels c0 + (k % cpt) * 8.
// (n_vt, cpg) = (4,8) (2,16) (1,32): 4 chunks; (2,8) (1,16): 2.  gamma / beta arrive pre-scaled by log2(e).
#ifdef TC_NO_FENCE
#define TC_SCHED_FENCE()
#else
#define TC_SCHED_FENCE() asm volatile("" ::: "memory")
#endif
// (Tried and dropped, twice: refilling the registers of every finished chunk with the same chunk of the NEXT half during the
// normalise pass, to hide its ~1 100 cycles of tensor-memory reads.  The reads slow the pass down by as much as they save.)
// `acc_bar` / `acc_parity`: the accumulator-full barrier of this half is waited for HERE, after the per-op set-up (masks, pointers:
// ~100 dependent instructions, ~700 cycles of a warp that shares its scheduler with three others) instead of before it, so the
// set-up runs under the MMAs.  `t_acc` (profiling build): clock after the wait.
__device__ __forceinline__ void epi_gn(const TcOp* o, const EpiCtx& cx, int h, uint32_t acc_bar, uint32_t acc_parity, long long* t_acc) {
  const int EPI = o->epi;
  const int q = cx.q, lane = cx.lane, b = lane & 7, sl = q * 4 + (lane >> 3);
  const int N = o->n, cpg = o->cpg, cpt = cpg >> 3, nch = o->n_vt * cpt;
  const int c0 = (h * 4 + cx.cq) * cpg;
  const int dst_pitch = o->dst_pitch, save_skip = o->save_skip, t_out = o->t_out;
  uint8_t* const dst_row = cx.arena + o->dst_off + 2048 + b * 128;     // + slot * 1024 + panel * pitch + swizzled chunk
  uint64_t v[4][4];
  uint32_t actm = 0, validm = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (k < nch) {
      const int vt = (cpt == 1) ? k : ((cpt == 2) ? (k >> 1) : 0);
      const int lo = o->tile_lo[vt], hi = o->tile_hi[vt];
      if (!(q * 4 + 4 <= lo || q * 4 >= hi)) actm |= 1u << k;           // warp-uniform: some row of this warp is valid
      if (sl >= lo && sl < hi) validm |= 1u << k;
    }
  }
  // ---- pass 1: conv bias, statistics over (time, channels of the group) per batch row.  Software pipeline over the chunks: the
  // tensor-memory read of chunk k + 1 (64 B / cycle for the whole SM, ~250 cycles per chunk with 16 warps reading) is in flight
  // while chunk k is summed (tcgen05.wait::ld waits for ALL outstanding loads, so the next one is issued right after the wait)
  auto load_chunk = [&](int k) {
    const int vt = (cpt == 1) ? k : ((cpt == 2) ? (k >> 1) : 0);
    uint32_t r[8];
    tmem_ld8(cx.lane_addr + vt * N + c0 + (k & (cpt - 1)) * 8, r);
    v[k][0] = pk2u(r[0], r[1]); v[k][1] = pk2u(r[2], r[3]); v[k][2] = pk2u(r[4], r[5]); v[k][3] = pk2u(r[6], r[7]);
  };
  mbar_wait(acc_bar, acc_parity);
  if (t_acc) *t_acc = clock64();
  tc_fence_after();
  if (cx.tl) cx.tl[3] = clock64();
  if (actm & 1u) load_chunk(0);
  uint64_t s2 = pk2(0.f, 0.f), ss2 = pk2(0.f, 0.f);
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    tmem_wait_ld();
    if (k == 0 && cx.tl) cx.tl[0] = clock64();
    if (k + 1 < 4 && ((actm >> (k + 1)) & 1u)) load_chunk(k + 1);
    if (!((actm >> k) & 1u)) continue;
    const int c = c0 + (k & (cpt - 1)) * 8;
    const float4 b0 = *reinterpret_cast<const float4*>(cx.par + c), b1 = *reinterpret_cast<const float4*>(cx.par + c + 4);
    const uint64_t u0 = add2(v[k][0], pk2(b0.x, b0.y)), u1 = add2(v[k][1], pk2(b0.z, b0.w));
    const uint64_t u2 = add2(v[k][2], pk2(b1.x, b1.y)), u3 = add2(v[k][3], pk2(b1.z, b1.w));
    v[k][0] = u0; v[k][1] = u1; v[k][2] = u2; v[k][3] = u3;
    if ((validm >> k) & 1u) {
      s2 = add2(s2, add2(add2(u0, u1), add2(u2, u3)));
      ss2 = add2(ss2, fma2(u0, u0, fma2(u1, u1, fma2(u2, u2, mul2(u3, u3)))));
    }
    TC_SCHED_FENCE();
  }
  float s, ss;
  {
    float a0, a1, q0, q1;
    upk2(s2, a0, a1); upk2(ss2, q0, q1);
    s = a0 + a1; ss = q0 + q1;
  }
  s += __shfl_xor_sync(0xffffffffu, s, 8);  ss += __shfl_xor_sync(0xffffffffu, ss, 8);
  s += __shfl_xor_sync(0xffffffffu, s, 16); ss += __shfl_xor_sync(0xffffffffu, ss, 16);
  float2* st = cx.st + (h & 1) * 128 + cx.cq * 32;          // [cq][quadrant][batch row]
  if (lane < 8) st[q * 8 + b] = make_float2(s, ss);
  if (cx.tl) cx.tl[1] = clock64();
  named_bar(2 + cx.cq, 128);                                // the 4 quadrant warps of this group
  if (cx.tl) cx.tl[2] = clock64();
  uint64_t rstd2, nmean2;
  {
    const float2 p0 = st[b], p1 = st[8 + b], p2 = st[16 + b], p3 = st[24 + b];   // fixed order: deterministic
    float S = ((p0.x + p1.x) + p2.x) + p3.x, SS = ((p0.y + p1.y) + p2.y) + p3.y;
    if (cx.tsplit) {                                          // the other half of the row (a + b is symmetric: both lanes get the same bits)
      const int bp = b ^ 4;
      const float2 r0 = st[bp], r1 = st[8 + bp], r2 = st[16 + bp], r3 = st[24 + bp];
      S += ((r0.x + r1.x) + r2.x) + r3.x; SS += ((r0.y + r1.y) + r2.y) + r3.y;
    }
    const float inv_n = __frcp_rn((float)((cx.tsplit ? 2 : 1) * t_out * cpg));
    const float mean = S * inv_n;
    const float var = fmaxf(SS * inv_n - mean * mean, 0.f);
    const float rstd = rsqrtf(var + 1e-5f);
    rstd2 = pk2(rstd, rstd); nmean2 = pk2(-mean, -mean);
  }
  // ---- pass 2: normalise / activate / add, write the next A operand
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (!((actm >> k) & 1u)) continue;
    const int vt = (cpt == 1) ? k : ((cpt == 2) ? (k >> 1) : 0);
    const int c = c0 + (k & (cpt - 1)) * 8;
    const bool valid = (validm >> k) & 1u;
    const int slot = o->tile_slot0[vt] + sl;
    uint64_t y[4];
    {
      const float4 g0 = *reinterpret_cast<const float4*>(cx.par + 256 + c), g1 = *reinterpret_cast<const float4*>(cx.par + 256 + c + 4);
      const float4 e0 = *reinterpret_cast<const float4*>(cx.par + 512 + c), e1 = *reinterpret_cast<const float4*>(cx.par + 512 + c + 4);
      const uint64_t gp[4] = {pk2(g0.x, g0.y), pk2(g0.z, g0.w), pk2(g1.x, g1.y), pk2(g1.z, g1.w)};
      const uint64_t ep[4] = {pk2(e0.x, e0.y), pk2(e0.z, e0.w), pk2(e1.x, e1.y), pk2(e1.z, e1.w)};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint64_t A = mul2(rstd2, gp[j]);
        const uint64_t B = fma2(nmean2, A, ep[j]);
        y[j] = mish2_log2(fma2(v[k][j], A, B));
      }
    }
    if (EPI == EPI_GN_TB) {
      const float4 t0 = *reinterpret_cast<const float4*>(cx.tb_s + b * TB_LD + c), t1 = *reinterpret_cast<const float4*>(cx.tb_s + b * TB_LD + c + 4);
      y[0] = add2(y[0], pk2(t0.x, t0.y)); y[1] = add2(y[1], pk2(t0.z, t0.w));
      y[2] = add2(y[2], pk2(t1.x, t1.y)); y[3] = add2(y[3], pk2(t1.z, t1.w));
    } else if (EPI == EPI_GN_RES_ACC) {
      uint32_t rr[8];
      tmem_ld8(cx.lane_addr + TC_RES_COL + vt * N + c, rr);
      tmem_wait_ld();
      const float4 s0 = *reinterpret_cast<const float4*>(cx.par + 768 + c), s1 = *reinterpret_cast<const float4*>(cx.par + 768 + c + 4);
      y[0] = add2(y[0], add2(pk2u(rr[0], rr[1]), pk2(s0.x, s0.y))); y[1] = add2(y[1], add2(pk2u(rr[2], rr[3]), pk2(s0.z, s0.w)));
      y[2] = add2(y[2], add2(pk2u(rr[4], rr[5]), pk2(s1.x, s1.y))); y[3] = add2(y[3], add2(pk2u(rr[6], rr[7]), pk2(s1.z, s1.w)));
    }
    if (valid) {
      const int sw = ((((c >> 3) & 7) ^ b) << 4);
      uint8_t* dp = dst_row + slot * 1024 + (c >> 6) * dst_pitch + sw;
      if (EPI == EPI_GN_RES_ID) {
        const uint4 old = *reinterpret_cast<const uint4*>(dp);
        y[0] = add2(y[0], pk2u(old.x << 16, old.x & 0xffff0000u)); y[1] = add2(y[1], pk2u(old.y << 16, old.y & 0xffff0000u));
        y[2] = add2(y[2], pk2u(old.z << 16, old.z & 0xffff0000u)); y[3] = add2(y[3], pk2u(old.w << 16, old.w & 0xffff0000u));
      }
      const uint4 pk = make_uint4(pack_bf16_2(y[0]), pack_bf16_2(y[1]), pack_bf16_2(y[2]), pack_bf16_2(y[3]));
      *reinterpret_cast<uint4*>(dp) = pk;
      if (cx.tsplit) store_inner_halo(cx.arena + o->dst_off + (c >> 6) * dst_pitch, t_out, slot, b, c, pk);
      if (save_skip >= 0)
        *reinterpret_cast<uint4*>(cx.skip_cta + save_skip + ((size_t)(c >> 6) * t_out + slot) * 1024 + b * 128 + sw) = pk;
    }
    TC_SCHED_FENCE();
  }
}

// bias-only epilogues (strided / transposed convolutions) and the final 1x1 convolution
__device__ __forceinline__ void epi_plain(const TcOp* o, const EpiCtx& cx, int h, const TcParams& P) {
  const int q = cx.q, lane = cx.lane, b = lane & 7, sl = q * 4 + (lane >> 3);
  const int N = o->n, nt = o->n_tiles, epi = o->epi;
  if (epi == EPI_OUT) {
    if (h != 0 || cx.cq != 0) return;
    const int row = row_of(cx.g, b, cx.tsplit);
    for (int vt = 0; vt < o->n_vt; ++vt) {
      const int lo = o->tile_lo[vt], hi = o->tile_hi[vt];
      if (q * 4 + 4 <= lo || q * 4 >= hi) continue;
      uint32_t r[8];
      tmem_ld8(cx.lane_addr + vt * N, r);
      tmem_wait_ld();
      const int slot = o->tile_slot0[vt] + sl;
      if (sl >= lo && sl < hi && row < cx.R) {
        float4 ov = make_float4(__uint_as_float(r[0]) + cx.par[0], __uint_as_float(r[1]) + cx.par[1],
                                __uint_as_float(r[2]) + cx.par[2], __uint_as_float(r[3]) + cx.par[3]);
        const size_t ti = cx.tsplit ? (size_t)row * 2 * P.T + (b >> 2) * P.T + slot : (size_t)row * P.T + slot;
        reinterpret_cast<float4*>(P.eps)[ti] = ov;
      }
    }
    return;
  }
  const int cw = N >> 3, c0 = (h * 4 + cx.cq) * cw;      // this warp's columns
  for (int vt = 0; vt < o->n_vt; ++vt) {
    const int mt = vt % nt, ph = vt / nt;
    const int lo = o->tile_lo[mt], hi = o->tile_hi[mt];
    if (q * 4 + 4 <= lo || q * 4 >= hi) continue;
    const bool valid = sl >= lo && sl < hi;
    const int slot = (epi == EPI_UP) ? 2 * (o->tile_slot0[mt] + sl) + ph : o->tile_slot0[mt] + sl;
    for (int c = c0; c < c0 + cw; c += 8) {
      uint32_t r[8];
      tmem_ld8(cx.lane_addr + vt * N + c, r);
      tmem_wait_ld();
      const float4 b0 = *reinterpret_cast<const float4*>(cx.par + c), b1 = *reinterpret_cast<const float4*>(cx.par + c + 4);
      const float y[8] = {__uint_as_float(r[0]) + b0.x, __uint_as_float(r[1]) + b0.y, __uint_as_float(r[2]) + b0.z,
                          __uint_as_float(r[3]) + b0.w, __uint_as_float(r[4]) + b1.x, __uint_as_float(r[5]) + b1.y,
                          __uint_as_float(r[6]) + b1.z, __uint_as_float(r[7]) + b1.w};
      store_chunk(o, cx, y, c, slot, b, valid);
    }
  }
}

// per-op parameters of op `o` for row group g -> shared memory (cp.async, one op ahead of use)
__device__ __forceinline__ void prefetch_params(const TcOp* o, const TcParams& P, float* par_buf, float* tb_s, int g, int etid) {
  const int cout = o->cout, q4 = cout >> 2;
  if (cout >= 64) {
    for (int i = etid; i < 4 * q4; i += TC_ETHREADS) {
      const int row = i / q4, c4 = i - row * q4;
      cp_async16(smem_u32(par_buf + row * 256 + c4 * 4), P.par + o->par_off + row * cout + c4 * 4);
    }
    if (o->epi == EPI_GN_TB) {
      for (int i = etid; i < q4; i += TC_ETHREADS) cp_async16(smem_u32(par_buf + 1024 + i * 4), P.tvec + o->tb_off + i * 4);
      for (int i = etid; i < TC_G * q4; i += TC_ETHREADS) {
        const int bb = i / q4, c4 = i - bb * q4;
        int r = row_of(g, bb, P.tsplit);
        r = r < P.R ? r : P.R - 1;
        cp_async16(smem_u32(tb_s + bb * TB_LD + c4 * 4), P.tbias + (size_t)r * P.tb_stride + o->tb_off + c4 * 4);
      }
    }
  } else if (etid < cout) {
    par_buf[etid] = P.par[o->par_off + etid];     // final 1x1 conv: cout = 4, bias only
  }
  cp_async_commit();
}

// ------------------------------------------------------------------------------------------------
// the kernel
// ------------------------------------------------------------------------------------------------
// PAIR: a cluster of two CTAs carries two row groups (8 rows each, one per CTA: activations, GroupNorm statistics, epilogue and skip
// buffers stay CTA-local) through the network in lock step.  Every MMA is ONE tcgen05.mma.cta_group::2 (M = 256: 128 GEMM rows per
// CTA) issued by the leader (rank 0); each CTA stages only HALF of the weight rows of a k-block (2-D TMA boxes of the weight blob,
// both CTAs' copies complete on the leader's full barrier), the instruction reads both halves.  The leader commits with a
// multicast arrive onto the ring-empty / accumulator-full barriers of both CTAs; the epilogue warps of both CTAs arrive on the
// leader's activation-ready barriers (remote mbarrier arrive for rank 1).
template <bool PROF, bool PAIR>
__global__ void __launch_bounds__(TC_THREADS, 1) unet_tc_kernel(const __grid_constant__ CUtensorMap tm8, const __grid_constant__ CUtensorMap tm16,
                                                                const __grid_constant__ CUtensorMap tm32, const __grid_constant__ CUtensorMap tm64,
                                                                const __grid_constant__ TcIssueTab IT,
                                                                const TcParams P) {
  constexpr int TC_SLOT = Ring<PAIR>::SLOT, TC_SLOTS = Ring<PAIR>::SLOTS;
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;
  const bool leader = rank == 0;
  // row groups: a single CTA walks g = blockIdx.x, += gridDim.x; a pair walks pair-groups and CTA `rank` takes group 2 * pg + rank
  const int unit0 = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x, unit_step = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const int n_units = PAIR ? (P.n_groups + 1) >> 1 : P.n_groups;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* arena = smem_raw;   // kept as a __shared__-space pointer so that ptxas emits LDS/STS, not generic LD/ST
  if ((smem_u32(smem_raw) & 1023u) != 0u) __trap();   // the swizzle atoms need 1024-byte alignment
  uint8_t* ring = arena + SM_RING;
  float* par_s = reinterpret_cast<float*>(arena + SM_PAR);
  float* tb_s = reinterpret_cast<float*>(arena + SM_TB);
  float2* st_s = reinterpret_cast<float2*>(arena + SM_ST);
  uint32_t* kbs_s = reinterpret_cast<uint32_t*>(arena + SM_KBS);
  uint64_t* bars = reinterpret_cast<uint64_t*>(arena + SM_BARS);
  TcShared* gsh = reinterpret_cast<TcShared*>(arena + SM_GLOB);
  uint32_t* tmem_slot = &gsh->tmem_base;
  // the warp index goes through a full-mask shuffle: the compiler then knows that the role branches below are warp-uniform and
  // keeps the issuer's / producer's loop state and descriptor arithmetic on the uniform datapath (the CUTLASS idiom)
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  const uint32_t bar_full = smem_u32(bars), bar_empty = smem_u32(bars + TC_UNITS);
  const uint32_t bar_act = smem_u32(bars + 2 * TC_UNITS), bar_acc = smem_u32(bars + 2 * TC_UNITS + 2);

  for (int i = tid; i < P.n_kbs; i += TC_THREADS) kbs_s[i] = P.kbs[i];
  if (tid == 0) {
    for (int i = 0; i < TC_UNITS; ++i) { mbar_init(bar_full + 8 * i, 1); mbar_init(bar_empty + 8 * i, 1); }
    mbar_init(bar_act, PAIR ? 2 * TC_EW : TC_EW); mbar_init(bar_act + 8, PAIR ? 2 * TC_EW : TC_EW);
    mbar_init(bar_acc, 1); mbar_init(bar_acc + 8, 1);
    fence_barrier_init();
    gsh->skip_cta = P.skipbuf + (size_t)blockIdx.x * P.skip_stride;
  }
  if (warp == TC_EW + 1) {
    if (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      tmem_alloc(smem_u32(tmem_slot), 512); tmem_relinquish();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();            // both CTAs' barriers exist before any remote arrive / remote complete_tx
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == TC_EW) {
    // ===================== weight producer =====================
    // every k-block takes one 16 KB ring slot; all lanes walk the loop, one elected lane issues the copy
    uint32_t par_empty = 0, slot_off = 0;
    int pos = 0;
    long long t_empty = 0;
    const uint32_t full0 = PAIR ? mapa_shared(bar_full, 0) : bar_full;       // pair: the leader's full barriers
    for (int g = unit0; g < n_units; g += unit_step) {
      const uint8_t* src = P.wblob + (size_t)(unit0 % P.wcopies) * P.wcopy_stride;
      int row = (unit0 % P.wcopies) * P.w_rows_per_copy;                     // pair: first blob row (128 B) of the k-block
      for (int k = 0; k < P.n_kbs; ++k) {
        const uint32_t kb = kbs_s[k];
        const uint32_t n8 = (kb >> 14) & 0x3Fu;
        const uint32_t bytes = n8 * (8u * 128u);                 // whole k-block (both halves in pair mode)
        if ((kb >> 26) & 1u) {
          // first k-block of a slot: wait for the slot, announce the bytes of the whole group
          uint32_t total = 0;
          for (int j = k; ; ++j) { const uint32_t kj = kbs_s[j]; total += ((kj >> 14) & 0x3Fu) * (8u * 128u); if ((kj >> 27) & 1u) break; }
          const long long tw0 = PROF ? clock64() : 0;
          mbar_wait(bar_empty + 8 * pos, ((par_empty >> pos) & 1u) ^ 1u);
          par_empty ^= 1u << pos;
          if (PROF) t_empty += clock64() - tw0;
          slot_off = 0;
          if (elect_one()) {
            if (PAIR) { if (leader) mbar_expect_tx_only(bar_full + 8 * pos, total); }
            else mbar_arrive_expect_tx(bar_full + 8 * pos, total);
          }
          __syncwarp();
        }
        if (elect_one()) {
          if (PAIR) {
            // this CTA's half of the weight rows: a box of N/2 rows starting at row + rank * N/2; completion on the leader's barrier
            const void* tm = n8 == 16u ? (const void*)&tm64 : (n8 == 8u ? (const void*)&tm32 : (n8 == 4u ? (const void*)&tm16 : (const void*)&tm8));
            tma2_load_2d(smem_u32(ring + pos * TC_SLOT) + slot_off, tm, 0, row + (int)(rank * n8 * 4u), full0 + 8 * pos);
          } else {
            bulk_g2s(smem_u32(ring + pos * TC_SLOT) + slot_off, src, bytes, bar_full + 8 * pos);
          }
        }
        __syncwarp();
        slot_off += PAIR ? bytes >> 1 : bytes;
        src += (size_t)(1u << ((kb >> 24) & 3)) * TC_UNIT;
        row += (int)(1u << ((kb >> 24) & 3)) * (TC_UNIT / 128);
        if ((kb >> 27) & 1u) pos = (pos + 1) & (TC_SLOTS - 1);
      }
    }
    if (PROF && lane == 0) { P.prof[blockIdx.x * 8 + 0] = t_empty; }
  } else if (warp == TC_EW + 1 && leader) {
    // ===================== MMA issuer (pair: the leader issues for both CTAs) =====================
    // all lanes walk the (warp-uniform) loop so that descriptors are computed on the uniform datapath; one elected
    // lane issues the tcgen05 instructions
    uint32_t par_full = 0, opn = 0, b_off = 0;
    int pos = 0;
    long long t_full = 0, t_act = 0, t_issue = 0, t_commit = 0;
    const long long t_start = PROF ? clock64() : 0;
    const uint32_t arena_u = smem_u32(arena), ring_u = smem_u32(ring);
    const uint32_t arena16 = arena_u >> 4, ring16 = ring_u >> 4;
    const uint32_t b_hi = (uint32_t)(make_desc_sw128(0, 1024) >> 32);
    for (int g = unit0; g < n_units; g += unit_step) {
      int kbi = 0;
      for (int oi = 0; oi < IT.n_ops; ++oi, ++opn) {
        const TcIssueOp& o = IT.op[oi];
        const int N = o.n, nt = o.nt, flags = o.flags;
        const int n_g0 = o.n_g0, n_g1 = o.n_g1, n_g2 = o.n_g2;
        const uint32_t a_hi = (uint32_t)(make_desc_sw128(0, (uint32_t)o.sbo) >> 32);
        const uint32_t ts0 = arena16 + (uint32_t)o.ts[0], ts1 = arena16 + (uint32_t)o.ts[1];
        const uint32_t ts2 = arena16 + (uint32_t)o.ts[2], ts3 = arena16 + (uint32_t)o.ts[3];
        // `count` k-blocks of an op with NT m-tiles (compile-time: no per-tile branches in the loop)
        auto issue_nt = [&](int count, auto nt_c) {
          constexpr int NT = decltype(nt_c)::value;
          for (int k = 0; k < count; ++k, ++kbi) {
            const uint4 rec = IT.kb[kbi];
            if (rec.w & KB_SLOT_FIRST) {                      // first k-block of a ring slot: its weights have landed?
              const long long tw0 = PROF ? clock64() : 0;
              mbar_wait(bar_full + 8 * pos, (par_full >> pos) & 1u);
              if (PROF) t_full += clock64() - tw0;
              par_full ^= 1u << pos;
              tc_fence_after();
              b_off = 0;
            }
            const uint32_t b_lo = ring16 + (uint32_t)pos * (TC_SLOT / 16) + b_off;
            const uint32_t b16 = rec.w >> 16, d_col = (rec.w >> 5) & 0x1FFu;
            b_off += (NT == 1 && (rec.w & KB_DUAL)) ? 2u * b16 : b16;
            const uint32_t acc = (rec.w >> 1) & 1u;
            const long long ti0 = PROF ? clock64() : 0;
            if (elect_one()) {
#pragma unroll
              for (int mt = 0; mt < NT; ++mt) {
                const uint32_t a_lo = rec.x + (mt == 0 ? ts0 : mt == 1 ? ts1 : mt == 2 ? ts2 : ts3);
                const uint32_t d_addr = tmem_base + d_col + mt * N;
                umma_lohi<PAIR>(d_addr, a_lo, a_hi, b_lo, b_hi, rec.z, acc);
                if (rec.w & KB_K4) {
                  umma_lohi<PAIR>(d_addr, a_lo + 2, a_hi, b_lo + 2, b_hi, rec.z, 1u);
                  umma_lohi<PAIR>(d_addr, a_lo + 4, a_hi, b_lo + 4, b_hi, rec.z, 1u);
                  umma_lohi<PAIR>(d_addr, a_lo + 6, a_hi, b_lo + 6, b_hi, rec.z, 1u);
                }
                if (NT == 1 && (rec.w & KB_DUAL)) {            // second k-block of the record (always 4 K steps, accumulating)
                  const uint32_t a1 = rec.y + ts0, b1 = b_lo + b16;
                  umma_lohi<PAIR>(d_addr, a1, a_hi, b1, b_hi, rec.z, 1u);
                  umma_lohi<PAIR>(d_addr, a1 + 2, a_hi, b1 + 2, b_hi, rec.z, 1u);
                  umma_lohi<PAIR>(d_addr, a1 + 4, a_hi, b1 + 4, b_hi, rec.z, 1u);
                  umma_lohi<PAIR>(d_addr, a1 + 6, a_hi, b1 + 6, b_hi, rec.z, 1u);
                }
              }
              if (rec.w & KB_SLOT_LAST) { if (PAIR) umma2_commit_pair(bar_empty + 8 * pos); else umma_commit(bar_empty + 8 * pos); }
            }
            __syncwarp();
            if (PROF) t_issue += clock64() - ti0;
            if (rec.w & KB_SLOT_LAST) pos = (pos + 1) & (TC_SLOTS - 1);
          }
        };
        auto issue = [&](int count) {
          if (nt == 1) issue_nt(count, std::integral_constant<int, 1>());
          else if (nt == 2) issue_nt(count, std::integral_constant<int, 2>());
          else if (nt == 3) issue_nt(count, std::integral_constant<int, 3>());
          else issue_nt(count, std::integral_constant<int, 4>());
        };
        auto commit = [&](uint32_t bar) {
          if (elect_one()) { if (PAIR) umma2_commit_pair(bar); else umma_commit(bar); }
          __syncwarp();
        };
        const uint32_t ph = opn & 1u;
        long long* tl = (PROF && blockIdx.x == 0 && g == unit0 && lane == 0) ? P.prof + gridDim.x * 8 + oi * 8 : nullptr;
        if (tl) tl[0] = clock64();
        long long tw1 = PROF ? clock64() : 0;
        mbar_wait(bar_act, ph);                                  // inputs written by half 0 of the previous epilogue
        if (!(flags & F_SPLIT_K)) mbar_wait(bar_act + 8, ph);
        if (PROF) t_act += clock64() - tw1;
        if (tl) tl[1] = clock64();
        tc_fence_after();
        issue(n_g0);
        if (flags & F_SPLIT_K) {
          tw1 = PROF ? clock64() : 0;
          mbar_wait(bar_act + 8, ph);
          if (PROF) t_act += clock64() - tw1;
          tc_fence_after();
        }
        issue(n_g1);
        if (flags & F_COMMIT_SPLIT) commit(bar_acc);
        issue(n_g2);
        if (!(flags & F_COMMIT_SPLIT)) commit(bar_acc);
        commit(bar_acc + 8);
        if (tl) tl[2] = clock64();
      }
    }
    if (PROF && lane == 0) { P.prof[blockIdx.x * 8 + 2] = t_full; P.prof[blockIdx.x * 8 + 3] = t_act; P.prof[blockIdx.x * 8 + 4] = clock64() - t_start; P.prof[blockIdx.x * 8 + 7] = t_issue; P.prof[blockIdx.x * 8 + 1] = t_commit; }
  } else if (warp < TC_EW) {
    // ===================== epilogue warps =====================
    EpiCtx cx;
    cx.etid = tid; cx.q = warp & 3; cx.cq = warp >> 2; cx.lane = lane;
    cx.arena = arena; cx.tb_s = tb_s; cx.st = st_s;
    cx.lane_addr = tmem_base + ((uint32_t)(cx.q * 32) << 16);
    cx.skip_cta = P.skipbuf + (size_t)blockIdx.x * P.skip_stride;
    cx.dbg_out = P.dbg_out; cx.dbg_stage = P.dbg_stage; cx.R = P.R; cx.tl = nullptr; cx.tsplit = P.tsplit;
    const int etid = cx.etid;
    uint32_t opn = 0;
    long long t_acc = 0;
    const long long t_start = PROF ? clock64() : 0;
    const uint32_t act0 = PAIR ? mapa_shared(bar_act, 0) : bar_act;          // pair: the leader's activation-ready barriers
    for (int u = unit0; u < n_units; u += unit_step) {
      const int g = PAIR ? 2 * u + (int)rank : u;
      cx.g = g;
      // ---- stage the latent x [8,T,4] fp32 as bf16 hi/lo channels 0..7 of panel 0 (region A, level 0)
      prefetch_params(IT.ops, P, par_s, tb_s, g, etid);
      if (P.tsplit) zero_halos_split(arena, P.zero0_offB, P.zero0_pitch, P.zero0_npanels, etid);
      else zero_halos(arena, P.zero0_offB, P.zero0_pitch, P.zero0_npanels, etid);
      // split-time mode: lane bb = half * 4 + row covers times [half * T, half * T + T); the slots -2, -1 / T, T + 1 of a lane are its
      // inner halo where the other half of the row continues (zero outside [0, 2T): those lines are the outer halo, zeroed above)
      const int t_lo = P.tsplit ? -2 : 0, t_n = P.tsplit ? P.T + 4 : P.T;
      for (int i = etid; i < t_n * TC_G; i += TC_ETHREADS) {
        const int t = (i >> 3) + t_lo, bb = i & 7, r = row_of(g, bb, P.tsplit);
        const int tg = P.tsplit ? (bb >> 2) * P.T + t : t, t_full = P.tsplit ? 2 * P.T : P.T;
        if (tg < 0 || tg >= t_full) continue;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r < P.R) v = reinterpret_cast<const float4*>(P.x)[(size_t)r * t_full + tg];
        float hx = __bfloat162float(__float2bfloat16_rn(v.x)), hy = __bfloat162float(__float2bfloat16_rn(v.y));
        float hz = __bfloat162float(__float2bfloat16_rn(v.z)), hw = __bfloat162float(__float2bfloat16_rn(v.w));
        uint4 c0 = make_uint4(pack_bf16(hx, hy), pack_bf16(hz, hw), pack_bf16(v.x - hx, v.y - hy), pack_bf16(v.z - hz, v.w - hw));
        uint8_t* rowp = arena + (t + 2) * 1024 + bb * 128;
        *reinterpret_cast<uint4*>(rowp + ((0 ^ bb) << 4)) = c0;
        *reinterpret_cast<uint4*>(rowp + ((1 ^ bb) << 4)) = make_uint4(0u, 0u, 0u, 0u);
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) {
        if (PAIR) { mbar_arrive_remote(act0); mbar_arrive_remote(act0 + 8); }
        else { mbar_arrive(bar_act); mbar_arrive(bar_act + 8); }
      }

      for (int oi = 0; oi < P.n_ops; ++oi, ++opn) {
        const TcOp* o = IT.ops + oi;
        cp_async_wait_all();
        epi_bar();                                   // parameters of this op are visible to every epilogue thread
        if (o->epi == EPI_GN_TB) {
          // fold the per-step time vector into the per-row cond bias: tb_s[b][c] += tvec[c]
          const float* tv = par_s + (oi & 1) * (PAR_ROWS * 256) + 1024;
          for (int i = etid; i < TC_G * o->cout; i += TC_ETHREADS) {
            const int bb = i / o->cout, c = i - bb * o->cout;
            tb_s[bb * TB_LD + c] += tv[c];
          }
          epi_bar();
        }
        if (oi + 1 < P.n_ops) prefetch_params(o + 1, P, par_s + ((oi + 1) & 1) * (PAR_ROWS * 256), tb_s, g, etid);
        cx.par = par_s + (oi & 1) * (PAR_ROWS * 256);
        const int epi = o->epi;
        const bool is_gn = (epi == EPI_GN_TB || epi == EPI_GN_RES_ACC || epi == EPI_GN_RES_ID || epi == EPI_GN);
#pragma unroll 1
        for (int h = 0; h < 2; ++h) {
          const long long tw0 = PROF ? clock64() : 0;
          long long* tl = (PROF && blockIdx.x == 0 && u == unit0 && etid == 0) ? P.prof + gridDim.x * 8 + oi * 8 : nullptr;
          cx.tl = (tl && h == 0) ? P.prof + (gridDim.x + TC_MAX_OPS) * 8 + oi * 4 : nullptr;
          if (is_gn) {
            epi_gn(o, cx, h, bar_acc + 8 * h, opn & 1u, tl ? tl + 3 + 2 * h : nullptr);
            if (PROF) t_acc += clock64() - tw0;
          } else {
            mbar_wait(bar_acc + 8 * h, opn & 1u);
            if (PROF) t_acc += clock64() - tw0;
            if (tl) tl[3 + 2 * h] = clock64();
            tc_fence_after();
            epi_plain(o, cx, h, P);
          }
          if (h == 1 && o->dbg_stage >= 0 && o->dbg_stage == P.dbg_stage && P.dbg_out != nullptr) {
            epi_bar();
            dump_stage(o, cx);
          }
          if (h == 1) {
            // ---- level change: zero the halo slots of the new layout; reload a skip connection
            if (o->zero_pitch) {
              if (P.tsplit) zero_halos_split(arena, o->zero_offB, o->zero_pitch, o->zero_npanels, etid);
              else zero_halos(arena, o->zero_offB, o->zero_pitch, o->zero_npanels, etid);
            }
            if (o->load_skip >= 0) {
              epi_bar();     // the skip stores of this CTA (possibly by this very op) are complete and visible
              const uint8_t* gp = cx.skip_cta + o->load_skip;
              const int per_panel = o->load_T * 64;          // uint4 per panel
              for (int i = etid; i < o->load_npanels * per_panel; i += TC_ETHREADS) {
                int p = i / per_panel, w = i - p * per_panel;
                *reinterpret_cast<uint4*>(arena + o->load_off + p * o->load_pitch + 2048 + w * 16) =
                    *reinterpret_cast<const uint4*>(gp + (size_t)i * 16);
              }
              if (P.tsplit) {
                // inner halos of the reloaded tensor, straight from the skip buffer: lane b >= 4 continues lane b - 4 (its last two
                // slots), lane b < 4 is continued by lane b + 4 (its first two slots); 16-byte chunk i of a lane sits at (i ^ lane)
                for (int i = etid; i < o->load_npanels * 128; i += TC_ETHREADS) {
                  const int ch = i & 7, bb = (i >> 3) & 7, j = (i >> 6) & 1, p = i >> 7;
                  const int bp = bb ^ 4, src_slot = bb >= 4 ? o->load_T - 2 + j : j, dst_slot = bb >= 4 ? j : o->load_T + 2 + j;
                  *reinterpret_cast<uint4*>(arena + o->load_off + p * o->load_pitch + dst_slot * 1024 + bb * 128 + ((ch ^ bb) << 4)) =
                      *reinterpret_cast<const uint4*>(gp + ((size_t)p * o->load_T + src_slot) * 1024 + bp * 128 + ((ch ^ bp) << 4));
                }
              }
            }
          }
          tc_fence_before();
          fence_proxy_async();
          __syncwarp();
          if (lane == 0 && oi + 1 < P.n_ops) {
            if (PAIR) mbar_arrive_remote(act0 + 8 * h); else mbar_arrive(bar_act + 8 * h);
          }
          if (tl) tl[4 + 2 * h] = clock64();
        }
      }
    }
    if (PROF && etid == 0) { P.prof[blockIdx.x * 8 + 5] = t_acc; P.prof[blockIdx.x * 8 + 6] = clock64() - t_start; }
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();            // nobody leaves (or frees tensor memory) while the peer may still touch this CTA
  if (warp == TC_EW + 1) {
    if (PAIR) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
    else tmem_dealloc(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------------
// weight packing: one k-block = [rows][64 k] bf16, 128B-swizzled image ready for a flat bulk copy
// ------------------------------------------------------------------------------------------------
__global__ void tc_pack_tile_kernel(uint8_t* __restrict__ dst, const float* __restrict__ w, int cout, int cin, int K,
                                    int transposed, int tap, int ci0, int n0, int rows, int dup4) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * 64) return;
  int nr = idx >> 6, k = idx & 63, n = n0 + nr;
  int ci = ci0 + k;
  if (dup4) ci = (k < 8) ? (k & 3) : cin;     // first layer: channels 0..3 = hi part, 4..7 = lo part of x
  float v = 0.f;
  if (n < cout && ci < cin) v = transposed ? w[((size_t)ci * cout + n) * K + tap] : w[((size_t)n * cin + ci) * K + tap];
  __nv_bfloat16 hv = __float2bfloat16_rn(v);
  *reinterpret_cast<__nv_bfloat16*>(dst + sw128_off(nr, k >> 3) + (k & 7) * 2) = hv;
}

__global__ void tc_copy_scale_kernel(float* __restrict__ dst, const float* __restrict__ src, int n, float scale) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[i] * scale;
}

static TcState* st_of(CldHandle* h) { return reinterpret_cast<TcState*>(h->tc); }

bool tc_level_layout(int horizon, TcLevel L[3]) {
  // 8-row mode covers 16..56 steps; above that each row runs as two lanes of horizon / 2 steps, which must be a multiple of 4 so
  // that every level of a lane has a whole number of slots
  const bool tsplit = horizon > 56;
  if (horizon < 16 || horizon % 4 || (tsplit && horizon % 8)) return false;
  const int T = tsplit ? horizon / 2 : horizon;
  const int np[3] = {1, 2, 4};
  for (int l = 0; l < 3; ++l) {
    TcLevel& v = L[l];
    v.T = T >> l; v.npanels = np[l];
    // 8-row mode: the 2 halo slots between two panels are shared (both zero); split-time mode: every panel has its own leading and
    // trailing halo, because the inner one carries the partner lane's edge slots
    if (tsplit) { v.pitch = (v.T + 4) * 1024; v.offB = np[l] * v.pitch; }
    else { v.pitch = (v.T + 2) * 1024; v.offB = np[l] * v.pitch + 2048; }
    v.n_tiles = (v.T + 15) / 16;
    for (int i = 0; i < 4; ++i) { v.slot0[i] = 0; v.lo[i] = 0; v.hi[i] = 0; }
    for (int i = 0; i < v.n_tiles; ++i) {
      bool last = i == v.n_tiles - 1;
      v.slot0[i] = (last && v.T >= 16) ? v.T - 16 : 16 * i;
      v.lo[i] = 16 * i - v.slot0[i];
      v.hi[i] = (v.T - v.slot0[i] < 16) ? v.T - v.slot0[i] : 16;
    }
    // every 16-slot tile read (plus taps, plus stride-2 reads from the level above) must stay inside the arena
    // (split-time mode: the regions fill the arena exactly; the reads of masked rows past its end land in the weight ring)
    if (tsplit ? (v.offB + v.npanels * v.pitch > TC_ARENA) : (v.offB + v.npanels * v.pitch + 5 * 1024 > TC_ARENA)) return false;
  }
  return true;
}

namespace {
using Level = TcLevel;

struct ConvSpec {          // one convolution (or one output phase of a transposed convolution)
  const float* w; int cout, cin, K, transposed;
  const int* tap_k; const int* tap_off; int ntaps;
  bool dup4;
};

struct Builder {
  TcState* s;
  size_t w_bytes = 0; size_t par_floats = 0;
  struct PackJob { size_t off; const float* w; int cout, cin, K, transposed, tap, ci0, n0, rows, dup4; };
  struct ParJob { size_t off; const float* src; int n; float scale; };
  std::vector<PackJob> packs; std::vector<ParJob> pars;

  int add_par(const float* bias, const float* gamma, const float* beta, const float* resb, int cout) {
    size_t off = par_floats;
    // GroupNorm gamma / beta are stored pre-scaled by log2(e): the epilogue evaluates Mish through 2^x
    const float* srcs[4] = {bias, gamma, beta, resb};
    const float scl[4] = {1.f, 1.4426950408889634f, 1.4426950408889634f, 1.f};
    for (int i = 0; i < 4; ++i) if (srcs[i]) pars.push_back({off + (size_t)i * cout, srcs[i], cout, scl[i]});
    par_floats += 4 * (size_t)((cout + 3) / 4 * 4);
    return (int)off;
  }
  // k-blocks of `cv` for output channels [n0, n0+rows) over the input panels panel_base[p0..p1): appended to the op
  int emit(const ConvSpec& cv, const int* panel_base, int p0, int p1, int n0, int rows, int acc_col, bool& first) {
    int count = 0;
    const int bytes = rows * 128;
    const int units = bytes <= TC_UNIT ? 1 : bytes / TC_UNIT;
    for (int t = 0; t < cv.ntaps; ++t)
      for (int p = p0; p < p1; ++p) {
        TcKb kb;
        kb.a_base = panel_base[p]; kb.shift = cv.tap_off[t] + 2;
        kb.w_off = (int)w_bytes;
        packs.push_back({w_bytes, cv.w, cv.cout, cv.cin, cv.K, cv.transposed, cv.tap_k[t], p * 64, n0, rows, cv.dup4 ? 1 : 0});
        w_bytes += (size_t)units * TC_UNIT;
        kb.acc_col = acc_col; kb.n = rows;
        kb.nk16 = cv.dup4 ? 1 : ((cv.cin - p * 64 >= 64) ? 4 : (cv.cin - p * 64 + 15) / 16);
        kb.first = first ? 1 : 0;
        kb.units = units; kb.slot_first = 1; kb.slot_last = 1;
        first = false;
        s->kbs.push_back(kb);
        ++count;
      }
    return count;
  }
};

void set_tiles(TcOp& o, const Level& L) {
  o.n_tiles = L.n_tiles;
  for (int i = 0; i < 4; ++i) { o.tile_slot0[i] = L.slot0[i]; o.tile_lo[i] = L.lo[i]; o.tile_hi[i] = L.hi[i]; }
}
TcOp blank_op() {
  TcOp o;
  memset(&o, 0, sizeof(o));
  o.sbo = 1024; o.slot_stride = 1; o.save_skip = -1; o.load_skip = -1; o.dbg_stage = -1; o.cpg = 8;
  return o;
}
}  // namespace

int tc_finalize(CldHandle* h, const float* const* p, cudaStream_t stream) {
  if (!h->tc) h->tc = new TcState();
  TcState* s = st_of(h);
  const CldConfig& c = h->cfg;
  const UnetLayout& sd = h->unet_layout;
  s->tsplit = c.horizon > 56;
  const int T = s->tsplit ? c.horizon / 2 : c.horizon;
  s->t_eff = T;
  Level L[3];
  if (!tc_level_layout(c.horizon, L)) return fail(h, CLD_ERR_UNSUPPORTED, "horizon too long for the bf16 arena");
  s->zero0_pitch = L[0].pitch; s->zero0_offB = L[0].offB;
  Builder B{s};
  s->ops.clear(); s->kbs.clear();
  const int k5[5] = {0, 1, 2, 3, 4}, o5[5] = {-2, -1, 0, 1, 2}, k1[1] = {0}, o1[1] = {0};
  const int k3[3] = {0, 1, 2}, o3[3] = {-1, 0, 1};
  const int kue[2] = {1, 3}, oue[2] = {0, -1}, kuo[2] = {0, 2}, ouo[2] = {1, 0};
  bool prev_commit_split = false;     // the previous op published its two output halves separately
  // ops with N >= split_min compute their output channels as two halves (epilogue of half 0 under the MMAs of half 1)
  int split_min = 128;      // measured: 256 -> 128 is -2 % on the launch (level 1), 64 gains nothing more (N = 32 MMAs cost what N = 64 ones do)
  if (const char* e = getenv("CLD_TC_SPLIT_MIN")) { int v = atoi(e); if (v == 64 || v == 128 || v == 256 || v == 512) split_min = v; }

  auto res_block = [&](int e, int lvl, const int* in_panels, int n_in, bool concat, int stage) {
    const BlkIdx& bk = sd.blk[e];
    const ResBlockW& rb = h->unet.rb[e];
    const Level& lv = L[lvl];
    const int N = rb.cout, half = N / 2;
    const bool has_res = bk.rw >= 0;
    const ConvSpec conv0{p[bk.c0w], N, rb.cin, 5, 0, k5, o5, 5, e == 0};
    const ConvSpec resc{has_res ? p[bk.rw] : nullptr, N, rb.cin, 1, 0, k1, o1, 1, e == 0};
    const ConvSpec conv1{p[bk.c1w], N, N, 5, 0, k5, o5, 5, false};
    // ---- op A: conv0 (+ residual 1x1 conv into the second accumulator set), GroupNorm + Mish + time bias
    // an M=128 MMA costs >= 64 cycles whatever its N (A-operand fetch), so only N = 256 layers are split into halves
    const bool csA = (N >= split_min) && !concat;    // concat blocks write h over x: the epilogue must wait for all MMAs
    const bool skA = csA && prev_commit_split && (n_in % 2 == 0);
    TcOp a = blank_op();
    a.n = N; set_tiles(a, lv); a.kb_first = (int)s->kbs.size();
    a.epi = EPI_GN_TB; a.cout = N; a.cpg = N / 8; a.t_out = lv.T; a.n_vt = lv.n_tiles;
    a.dst_off = concat ? 0 : lv.offB; a.dst_pitch = lv.pitch;
    a.par_off = B.add_par(p[bk.c0b], p[bk.g0], p[bk.b0], nullptr, N); a.tb_off = rb.tb_off;
    a.flags = (csA ? F_COMMIT_SPLIT : 0) | (skA ? F_SPLIT_K : 0);
    if (csA) {
      bool f0 = true, f1 = true, fr0 = true, fr1 = true;
      if (skA) {
        a.n_g0 = B.emit(conv0, in_panels, 0, n_in / 2, 0, half, 0, f0);
        a.n_g1 = B.emit(conv0, in_panels, n_in / 2, n_in, 0, half, 0, f0);
      } else {
        a.n_g1 = B.emit(conv0, in_panels, 0, n_in, 0, half, 0, f0);
      }
      a.n_g2 = B.emit(conv0, in_panels, 0, n_in, half, half, half, f1);
      if (has_res) {
        a.n_g2 += B.emit(resc, in_panels, 0, n_in, 0, half, TC_RES_COL, fr0);
        a.n_g2 += B.emit(resc, in_panels, 0, n_in, half, half, TC_RES_COL + half, fr1);
      }
    } else {
      bool f0 = true, fr = true;
      a.n_g0 = B.emit(conv0, in_panels, 0, n_in, 0, N, 0, f0);
      if (has_res) a.n_g0 += B.emit(resc, in_panels, 0, n_in, 0, N, TC_RES_COL, fr);
    }
    s->ops.push_back(a);
    // ---- op B: conv1, GroupNorm + Mish + residual
    const bool csB = (N >= split_min) && !concat;     // concat blocks run conv1 in place (h and the output share region A)
    const bool skB = csB && csA;                      // h has N/64 >= 2 panels
    TcOp b = blank_op();
    b.n = N; set_tiles(b, lv); b.kb_first = (int)s->kbs.size();
    b.epi = has_res ? EPI_GN_RES_ACC : EPI_GN_RES_ID; b.cout = N; b.cpg = N / 8; b.t_out = lv.T; b.n_vt = lv.n_tiles;
    b.dst_off = 0; b.dst_pitch = lv.pitch;
    b.par_off = B.add_par(p[bk.c1b], p[bk.g1], p[bk.b1], has_res ? p[bk.rb] : nullptr, N);
    b.flags = (csB ? F_COMMIT_SPLIT : 0) | (skB ? F_SPLIT_K : 0);
    int hp[4];
    const int nhp = N / 64;
    for (int p = 0; p < nhp; ++p) hp[p] = a.dst_off + p * lv.pitch;
    if (csB) {
      bool f0 = true, f1 = true;
      if (skB) {
        b.n_g0 = B.emit(conv1, hp, 0, nhp / 2, 0, half, 0, f0);
        b.n_g1 = B.emit(conv1, hp, nhp / 2, nhp, 0, half, 0, f0);
      } else {
        b.n_g1 = B.emit(conv1, hp, 0, nhp, 0, half, 0, f0);
      }
      b.n_g2 = B.emit(conv1, hp, 0, nhp, half, half, half, f1);
    } else {
      bool f0 = true;
      b.n_g0 = B.emit(conv1, hp, 0, nhp, 0, N, 0, f0);
    }
    b.dbg_stage = stage;
    s->ops.push_back(b);
    prev_commit_split = csB;
  };
  // strided / transposed convolution between levels (bias-only epilogue, unsplit)
  auto resample = [&](bool up, int ch, const float* w, const float* bias, const Level& lin, const Level& lout, const int* in_panels,
                      int n_in, int stage) -> TcOp& {
    TcOp d = blank_op();
    d.n = ch; d.kb_first = (int)s->kbs.size();
    d.cout = ch; d.t_out = lout.T; d.dst_off = 0; d.dst_pitch = lout.pitch;
    d.par_off = B.add_par(bias, nullptr, nullptr, nullptr, ch);
    d.zero_pitch = lout.pitch; d.zero_npanels = lout.npanels; d.zero_offB = lout.offB; d.dbg_stage = stage;
    if (!up) {
      set_tiles(d, lout); d.sbo = 2048; d.slot_stride = 2; d.epi = EPI_BIAS; d.n_vt = lout.n_tiles;
      const ConvSpec cv{w, ch, ch, 3, 0, k3, o3, 3, false};
      bool f = true;
      d.n_g0 = B.emit(cv, in_panels, 0, n_in, 0, ch, 0, f);
    } else {
      set_tiles(d, lin); d.epi = EPI_UP; d.n_vt = 2 * lin.n_tiles;
      const ConvSpec ce{w, ch, ch, 4, 1, kue, oue, 2, false}, co{w, ch, ch, 4, 1, kuo, ouo, 2, false};
      bool fe = true, fo = true;
      d.n_g0 = B.emit(ce, in_panels, 0, n_in, 0, ch, 0, fe);
      d.n_g0 += B.emit(co, in_panels, 0, n_in, 0, ch, lin.n_tiles * ch, fo);
    }
    s->ops.push_back(d);
    prev_commit_split = false;
    return s->ops.back();
  };
  auto panels_of = [&](int off, int pitch, int n, int* out) { for (int p = 0; p < n; ++p) out[p] = off + p * pitch; };
  const int skip1_off = 0, skip1_bytes = 2 * L[1].T * 1024, skip2_off = skip1_bytes, skip2_bytes = 4 * L[2].T * 1024;
  int pa[8];

  // level 0
  panels_of(0, L[0].pitch, 1, pa); res_block(0, 0, pa, 1, false, 0);
  res_block(1, 0, pa, 1, false, 1);
  resample(false, 64, p[sd.down[0][0]], p[sd.down[0][1]], L[0], L[1], pa, 1, 2);
  // level 1
  panels_of(0, L[1].pitch, 1, pa); res_block(2, 1, pa, 1, false, 3);
  panels_of(0, L[1].pitch, 2, pa); res_block(3, 1, pa, 2, false, 4);
  s->ops.back().save_skip = skip1_off;
  resample(false, 128, p[sd.down[1][0]], p[sd.down[1][1]], L[1], L[2], pa, 2, 5);
  // level 2
  panels_of(0, L[2].pitch, 2, pa); res_block(4, 2, pa, 2, false, 6);
  panels_of(0, L[2].pitch, 4, pa); res_block(5, 2, pa, 4, false, 7);
  s->ops.back().save_skip = skip2_off;
  res_block(6, 2, pa, 4, false, 8);
  res_block(7, 2, pa, 4, false, 9);
  {  // after mid_block2: bring skip2 back into region B
    TcOp& o = s->ops.back();
    o.load_skip = skip2_off; o.load_off = L[2].offB; o.load_pitch = L[2].pitch; o.load_npanels = 4; o.load_T = L[2].T;
  }
  panels_of(0, L[2].pitch, 4, pa); panels_of(L[2].offB, L[2].pitch, 4, pa + 4);
  prev_commit_split = false;
  res_block(8, 2, pa, 8, true, 10);
  panels_of(0, L[2].pitch, 2, pa); res_block(9, 2, pa, 2, false, 11);
  {  // ups.0.2: transposed conv 128 -> 128, level 2 -> level 1 (two output phases); then skip1 into region B
    TcOp& u = resample(true, 128, p[sd.up[0][0]], p[sd.up[0][1]], L[2], L[1], pa, 2, 12);
    u.load_skip = skip1_off; u.load_off = L[1].offB; u.load_pitch = L[1].pitch; u.load_npanels = 2; u.load_T = L[1].T;
  }
  // level 1 (up path)
  panels_of(0, L[1].pitch, 2, pa); panels_of(L[1].offB, L[1].pitch, 2, pa + 2);
  res_block(10, 1, pa, 4, true, 13);
  panels_of(0, L[1].pitch, 1, pa); res_block(11, 1, pa, 1, false, 14);
  resample(true, 64, p[sd.up[1][0]], p[sd.up[1][1]], L[1], L[0], pa, 1, 15);
  {  // final_conv.0: conv k5 + GroupNorm + Mish -> region B ; final_conv.1: 1x1 conv 64 -> 4 -> eps
    panels_of(0, L[0].pitch, 1, pa);
    TcOp f = blank_op();
    f.n = 64; set_tiles(f, L[0]); f.kb_first = (int)s->kbs.size();
    f.epi = EPI_GN; f.cout = 64; f.cpg = 8; f.t_out = L[0].T; f.n_vt = L[0].n_tiles; f.dst_off = L[0].offB; f.dst_pitch = L[0].pitch;
    f.par_off = B.add_par(p[sd.fin[1]], p[sd.fin[2]], p[sd.fin[3]], nullptr, 64); f.dbg_stage = 16;
    const ConvSpec cf{p[sd.fin[0]], 64, 64, 5, 0, k5, o5, 5, false};
    bool ff = true;
    f.n_g0 = B.emit(cf, pa, 0, 1, 0, 64, 0, ff);
    s->ops.push_back(f);
    TcOp g = blank_op();
    g.n = 16; set_tiles(g, L[0]); g.kb_first = (int)s->kbs.size();
    g.epi = EPI_OUT; g.cout = 4; g.t_out = L[0].T; g.n_vt = L[0].n_tiles;
    g.par_off = B.add_par(p[sd.fin[5]], nullptr, nullptr, nullptr, 4);
    panels_of(L[0].offB, L[0].pitch, 1, pa);
    const ConvSpec cg{p[sd.fin[4]], 4, 64, 1, 0, k1, o1, 1, false};
    bool fg = true;
    g.n_g0 = B.emit(cg, pa, 0, 1, 0, 16, 0, fg);
    s->ops.push_back(g);
  }
  // accumulators must fit their half of the 512 TMEM columns
  for (const TcOp& o : s->ops)
    if (o.n_vt * o.n > TC_RES_COL) return fail(h, CLD_ERR_UNSUPPORTED, "accumulators exceed tensor memory");
  if (s->ops.size() > (size_t)TC_MAX_OPS || s->kbs.size() > (size_t)TC_MAX_KBS)
    return fail(h, CLD_ERR_UNSUPPORTED, "op table too large (%zu ops, %zu k-blocks)", s->ops.size(), s->kbs.size());

  // ---- materialise blobs on the device
  auto alloc = [&](void** p, size_t bytes) -> int {
    CLD_CUDA_OK(h, cudaMalloc(p, bytes));
    h->allocs.push_back(*p);
    return 0;
  };
  int rc;
  s->wblob_bytes = B.w_bytes; s->par_floats = B.par_floats;
  // every CTA streams the same bytes at about the same time; replicas at different addresses spread the
  // requests over more L2 slices (the set fits L2 many times over)
  s->wcopies = 8;
  if (const char* e = getenv("CLD_TC_WCOPIES")) { int v = atoi(e); if (v >= 1 && v <= 16) s->wcopies = v; }
  if ((rc = alloc((void**)&s->wblob, B.w_bytes * s->wcopies))) return rc;
  if ((rc = alloc((void**)&s->par, B.par_floats * sizeof(float)))) return rc;
  if ((rc = alloc((void**)&s->zeros, CLD_TB_TOTAL_MAX * sizeof(float)))) return rc;
  CLD_CUDA_OK(h, cudaMemsetAsync(s->wblob, 0, B.w_bytes, stream));
  CLD_CUDA_OK(h, cudaMemsetAsync(s->par, 0, B.par_floats * sizeof(float), stream));
  CLD_CUDA_OK(h, cudaMemsetAsync(s->zeros, 0, CLD_TB_TOTAL_MAX * sizeof(float), stream));
  for (const auto& j : B.packs) {
    tc_pack_tile_kernel<<<(j.rows * 64 + 255) / 256, 256, 0, stream>>>(s->wblob + j.off, j.w, j.cout, j.cin, j.K, j.transposed,
                                                                      j.tap, j.ci0, j.n0, j.rows, j.dup4);
  }
  CLD_LAUNCH_OK(h, "tc_pack_tile_kernel");
  for (int cpy = 1; cpy < s->wcopies; ++cpy)
    CLD_CUDA_OK(h, cudaMemcpyAsync(s->wblob + (size_t)cpy * B.w_bytes, s->wblob, B.w_bytes, cudaMemcpyDeviceToDevice, stream));
  for (const auto& j : B.pars) tc_copy_scale_kernel<<<(j.n + 255) / 256, 256, 0, stream>>>(s->par + j.off, j.src, j.n, j.scale);
  CLD_LAUNCH_OK(h, "tc_copy_scale_kernel");
  // ring-slot groups: consecutive k-blocks of one issue group (G0 | G1 | G2 of an op) with the same N share a slot while their
  // bytes (per CTA: half the rows in pair mode) fit; a k-block smaller than a 4 KB unit is not contiguous with its successor
  s->pair = true;
  if (const char* e = getenv("CLD_TC_PAIR")) s->pair = atoi(e) != 0;
  {
    int max_group = 8;
    if (const char* e = getenv("CLD_TC_KBGROUP")) { int v = atoi(e); if (v >= 1 && v <= 8) max_group = v; }
    for (const TcOp& o : s->ops) {
      const int lens[3] = {o.n_g0, o.n_g1, o.n_g2};
      int k = o.kb_first;
      for (int gi = 0; gi < 3; ++gi) {
        const int end = k + lens[gi];
        while (k < end) {
          const int n = s->kbs[k].n;
          const int per_cta = s->pair ? n * 64 : n * 128;
          int cnt = 1;
          while (k + cnt < end && cnt < max_group && s->kbs[k + cnt].n == n && n * 128 >= TC_UNIT && (cnt + 1) * per_cta <= Ring<true>::SLOT) ++cnt;
          for (int j = 0; j < cnt; ++j) { s->kbs[k + j].slot_first = j == 0; s->kbs[k + j].slot_last = j == cnt - 1; }
          k += cnt;
        }
      }
    }
  }
  std::vector<uint32_t> packed(s->kbs.size());
  size_t expect_off = 0;
  for (size_t k = 0; k < s->kbs.size(); ++k) {
    const TcKb& kb = s->kbs[k];
    if ((size_t)kb.w_off != expect_off || kb.a_base % 1024 || kb.acc_col % 8 || kb.n % 8)
      return fail(h, CLD_ERR_UNSUPPORTED, "internal: k-block record not packable");
    expect_off += (size_t)kb.units * TC_UNIT;
    uint32_t a_slots = (uint32_t)(kb.a_base / 1024 + kb.shift);
    int ul = kb.units == 1 ? 0 : kb.units == 2 ? 1 : kb.units == 4 ? 2 : kb.units == 8 ? 3 : -1;
    if (a_slots > 255u || kb.acc_col > 504 || kb.nk16 > 4 || kb.n > 256 || ul < 0 || kb.units * TC_UNIT > Ring<false>::SLOT)
      return fail(h, CLD_ERR_UNSUPPORTED, "internal: k-block field overflow");
    packed[k] = a_slots | ((uint32_t)(kb.acc_col / 8) << 8) | ((uint32_t)(kb.n / 8) << 14) | ((uint32_t)kb.nk16 << 20) |
                ((uint32_t)kb.first << 23) | ((uint32_t)ul << 24) | ((uint32_t)kb.slot_first << 26) | ((uint32_t)kb.slot_last << 27);
  }
  {
    size_t next = 0;
    for (const TcOp& o : s->ops) {
      if ((size_t)o.kb_first != next) return fail(h, CLD_ERR_UNSUPPORTED, "internal: k-blocks of the ops are not consecutive");
      next += (size_t)(o.n_g0 + o.n_g1 + o.n_g2);
    }
    if (next != s->kbs.size()) return fail(h, CLD_ERR_UNSUPPORTED, "internal: op k-block range");
  }
  if (!s->itab) s->itab = new TcIssueTab();
  memset(s->itab, 0, sizeof(TcIssueTab));
  s->itab->n_ops = (int)s->ops.size(); s->itab->n_kbs = (int)s->kbs.size();
  for (size_t i = 0; i < s->ops.size(); ++i) {
    const TcOp& o = s->ops[i];
    TcIssueOp& d = s->itab->op[i];
    s->itab->ops[i] = o;
    d.n_g0 = o.n_g0; d.n_g1 = o.n_g1; d.n_g2 = o.n_g2; d.flags = o.flags; d.n = o.n; d.nt = o.n_tiles; d.sbo = o.sbo;
    for (int t = 0; t < 4; ++t) d.ts[t] = o.tile_slot0[t] * o.slot_stride * 64;
  }
  {
    int dual = 1;
    if (const char* e = getenv("CLD_TC_DUAL")) dual = atoi(e) != 0;
    int nrec = 0;
    for (size_t i = 0; i < s->ops.size(); ++i) {
      const TcOp& o = s->ops[i];
      TcIssueOp& d = s->itab->op[i];
      const int lens[3] = {o.n_g0, o.n_g1, o.n_g2};
      int* out_len[3] = {&d.n_g0, &d.n_g1, &d.n_g2};
      int k = o.kb_first;
      for (int gi = 0; gi < 3; ++gi) {
        const int end = k + lens[gi];
        int cnt = 0;
        while (k < end) {
          const TcKb& kb = s->kbs[k];
          if (kb.nk16 != 1 && kb.nk16 != 4) return fail(h, CLD_ERR_UNSUPPORTED, "internal: k-block with %d K=16 steps", kb.nk16);
          const uint32_t per_cta16 = (uint32_t)(s->pair ? kb.n * 64 : kb.n * 128) / 16u;
          uint4 r;
          r.x = (uint32_t)(kb.a_base / 1024 + kb.shift) * 64u;
          r.y = 0;
          r.z = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(kb.n >> 3) << 17) | ((uint32_t)((s->pair ? 256 : 128) >> 4) << 24);
          r.w = (kb.nk16 == 4 ? KB_K4 : 0u) | (kb.first ? 0u : KB_ACC) | (kb.slot_first ? KB_SLOT_FIRST : 0u) | ((uint32_t)kb.acc_col << 5) | (per_cta16 << 16);
          bool last = kb.slot_last;
          int used = 1;
          if (dual && o.n_tiles == 1 && !kb.slot_last && k + 1 < end) {
            const TcKb& k2 = s->kbs[k + 1];
            if (kb.nk16 == 4 && k2.nk16 == 4 && !k2.first && k2.acc_col == kb.acc_col && k2.n == kb.n && !k2.slot_first) {
              r.y = (uint32_t)(k2.a_base / 1024 + k2.shift) * 64u;
              r.w |= KB_DUAL;
              last = k2.slot_last;
              used = 2;
            }
          }
          if (last) r.w |= KB_SLOT_LAST;
          if (nrec >= TC_MAX_KBS) return fail(h, CLD_ERR_UNSUPPORTED, "internal: issuer table overflow");
          s->itab->kb[nrec++] = r;
          k += used; ++cnt;
        }
        *out_len[gi] = cnt;
      }
    }
    s->itab->n_kbs = nrec;
  }
  if ((rc = alloc((void**)&s->d_ops, s->ops.size() * sizeof(TcOp)))) return rc;
  if ((rc = alloc((void**)&s->d_kbs, packed.size() * sizeof(uint32_t)))) return rc;
  CLD_CUDA_OK(h, cudaMemcpyAsync(s->d_ops, s->ops.data(), s->ops.size() * sizeof(TcOp), cudaMemcpyHostToDevice, stream));
  CLD_CUDA_OK(h, cudaMemcpyAsync(s->d_kbs, packed.data(), packed.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
  CLD_CUDA_OK(h, cudaStreamSynchronize(stream));
  s->grid = h->num_sms;
  s->skip_stride = ((skip1_bytes + skip2_bytes + 1023) / 1024) * 1024;
  if ((rc = alloc((void**)&s->skipbuf, (size_t)s->grid * s->skip_stride))) return rc;
  if (getenv("CLD_TC_PROF")) {
    if ((rc = alloc((void**)&s->prof, (size_t)(s->grid + 2 * TC_MAX_OPS) * 8 * sizeof(long long)))) return rc;
    CLD_CUDA_OK(h, cudaMemsetAsync(s->prof, 0, (size_t)(s->grid + 2 * TC_MAX_OPS) * 8 * sizeof(long long), stream));
  }
  CLD_CUDA_OK(h, cudaFuncSetAttribute(unet_tc_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM));
  CLD_CUDA_OK(h, cudaFuncSetAttribute(unet_tc_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM));
  CLD_CUDA_OK(h, cudaFuncSetAttribute(unet_tc_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM));
  CLD_CUDA_OK(h, cudaFuncSetAttribute(unet_tc_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM));
  // CTA-pair kernel (default): the weight blob (all replicas) as a 2-D tensor of 128-byte rows; a box = the half of a k-block
  // one CTA stages (N/2 = 8, 32 or 64 rows).  The blob is already swizzled, so the copies are flat (SWIZZLE_NONE).
  memset(&s->tm8, 0, sizeof(CUtensorMap)); memset(&s->tm16, 0, sizeof(CUtensorMap)); memset(&s->tm32, 0, sizeof(CUtensorMap)); memset(&s->tm64, 0, sizeof(CUtensorMap));
  if (s->pair) {
    typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                      const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn)
      return fail(h, CLD_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
    if (B.w_bytes % 128) return fail(h, CLD_ERR_UNSUPPORTED, "internal: weight blob is not a whole number of 128-byte rows");
    CUtensorMap* maps[4] = {&s->tm8, &s->tm16, &s->tm32, &s->tm64};
    const cuuint32_t rows[4] = {8, 16, 32, 64};
    for (int i = 0; i < 4; ++i) {
      cuuint64_t dims[2] = {64, (cuuint64_t)(B.w_bytes / 128) * (cuuint64_t)s->wcopies};
      cuuint64_t strides[1] = {128};
      cuuint32_t box[2] = {64, rows[i]}, es[2] = {1, 1};
      const CUresult r = ((EncodeTiledFn)fn)(maps[i], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void*)s->wblob, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                             CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) return fail(h, CLD_ERR_CUDA, "cuTensorMapEncodeTiled rejected the weight tensor (box of %u rows): %d", rows[i], (int)r);
    }
    for (const TcKb& kb : s->kbs)
      if (kb.n != 16 && kb.n != 32 && kb.n != 64 && kb.n != 128) return fail(h, CLD_ERR_UNSUPPORTED, "internal: k-block of %d weight rows has no pair box", kb.n);
  }
  CLD_CUDA_OK(h, cudaStreamSynchronize(stream));
  s->ready = true;
  (void)skip2_off;
  return 0;
}

// time / cond projection shared with the fp32 path (kernels_unet_fp32.cu)
int unet_time_bias(CldHandle* h, const float* cond, const int64_t* t, int R, cudaStream_t s);

static int tc_launch(CldHandle* h, const float* x, float* eps, int R, const float* tvec, cudaStream_t stream);

int tc_unet_forward(CldHandle* h, const float* x, const float* cond, const int64_t* t, float* eps, int R, cudaStream_t stream) {
  TcState* s = st_of(h);
  if (!s || !s->ready) return fail(h, CLD_ERR_STATE, "bf16 denoiser weights not packed");
  int rc;
  if ((rc = unet_time_bias(h, cond, t, R, stream))) return rc;
  return tc_launch(h, x, eps, R, s->zeros, stream);
}

int tc_unet_forward_prepared(CldHandle* h, const float* x, float* eps, int R, cudaStream_t stream, const float* tvec) {
  TcState* s = st_of(h);
  if (!s || !s->ready) return fail(h, CLD_ERR_STATE, "bf16 denoiser weights not packed");
  return tc_launch(h, x, eps, R, tvec ? tvec : h->tvec, stream);
}

static int tc_launch(CldHandle* h, const float* x, float* eps, int R, const float* tvec, cudaStream_t stream) {
  TcState* s = st_of(h);
  TcParams P;
  P.tvec = tvec;
  P.ops = s->d_ops; P.n_ops = (int)s->ops.size(); P.kbs = s->d_kbs; P.n_kbs = (int)s->kbs.size(); P.wblob = s->wblob; P.wcopy_stride = s->wblob_bytes; P.wcopies = s->wcopies; P.par = s->par;
  P.w_rows_per_copy = (int)(s->wblob_bytes / 128);
  P.tbias = h->tbias; P.tb_stride = h->unet.tb_total; P.x = x; P.eps = eps; P.R = R; P.T = s->t_eff; P.tsplit = s->tsplit ? 1 : 0;
  const int rows_per_group = s->tsplit ? 4 : TC_G;
  P.n_groups = (R + rows_per_group - 1) / rows_per_group; P.skipbuf = s->skipbuf; P.skip_stride = s->skip_stride;
  P.zero0_pitch = s->zero0_pitch; P.zero0_npanels = 1; P.zero0_offB = s->zero0_offB;
  P.dbg_stage = h->dbg_out ? h->dbg_stage : -1; P.dbg_out = h->dbg_out;
  P.prof = s->prof;
  int grid = P.n_groups < s->grid ? P.n_groups : s->grid;
  if (s->pair) {
    const int n_pairs = (P.n_groups + 1) / 2, clusters = n_pairs < s->grid / 2 ? n_pairs : s->grid / 2;
    grid = 2 * clusters;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(TC_THREADS); cfg.dynamicSmemBytes = TC_SMEM; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    cudaError_t e = s->prof ? cudaLaunchKernelEx(&cfg, unet_tc_kernel<true, true>, s->tm8, s->tm16, s->tm32, s->tm64, *s->itab, P)
                            : cudaLaunchKernelEx(&cfg, unet_tc_kernel<false, true>, s->tm8, s->tm16, s->tm32, s->tm64, *s->itab, P);
    if (e != cudaSuccess) return fail(h, CLD_ERR_CUDA, "launch of unet_tc_kernel (pair) failed: %s", cudaGetErrorString(e));
  } else if (s->prof) {
    unet_tc_kernel<true, false><<<grid, TC_THREADS, TC_SMEM, stream>>>(s->tm8, s->tm16, s->tm32, s->tm64, *s->itab, P);
  } else {
    unet_tc_kernel<false, false><<<grid, TC_THREADS, TC_SMEM, stream>>>(s->tm8, s->tm16, s->tm32, s->tm64, *s->itab, P);
  }
  CLD_LAUNCH_OK(h, "unet_tc_kernel");
  if (s->prof) {
    // debug only (CLD_TC_PROF=1): per-CTA cycle counters of the three roles, printed for CTA 0 and averaged
    std::vector<long long> hp((size_t)(grid + 2 * TC_MAX_OPS) * 8);
    CLD_CUDA_OK(h, cudaStreamSynchronize(stream));
    CLD_CUDA_OK(h, cudaMemcpy(hp.data(), s->prof, hp.size() * sizeof(long long), cudaMemcpyDeviceToHost));
    double avg[8] = {0};
    for (int b = 0; b < grid; ++b) for (int i = 0; i < 8; ++i) avg[i] += (double)hp[(size_t)b * 8 + i] / grid;
    fprintf(stderr, "[tc prof] producer: wait_empty %.0f | mma: wait_full %.0f wait_act %.0f issue %.0f commit %.0f of %.0f | epilogue: wait_acc %.0f of %.0f cycles\n",
            avg[0], avg[2], avg[3], avg[7], avg[1], avg[4], avg[5], avg[6]);
    if (getenv("CLD_TC_TIMELINE")) {
      const long long* tl = hp.data() + (size_t)grid * 8;
      const long long t0 = tl[0];
      for (size_t oi = 0; oi < s->ops.size(); ++oi) {
        const long long* r = tl + oi * 8;
        const TcOp& o = s->ops[oi];
        fprintf(stderr, "[tc op %2zu epi %d N %3d nvt %d kb %3d fl %d] mma: start %7lld act_ok %7lld done %7lld (issue %6lld) | epi h0: acc %7lld end %7lld (%6lld) h1: acc %7lld end %7lld (%6lld)\n",
                oi, o.epi, o.n, o.n_vt, o.n_g0 + o.n_g1 + o.n_g2, o.flags, r[0] - t0, r[1] - t0, r[2] - t0, r[2] - r[1], r[3] - t0, r[4] - t0, r[4] - r[3],
                r[5] - t0, r[6] - t0, r[6] - r[5]);
        const long long* e = hp.data() + (size_t)(grid + TC_MAX_OPS) * 8 + oi * 4;
        if (e[0]) fprintf(stderr, "      item h0 warp0: acc->first load issued %lld | -> loaded %lld | pass1 %lld | bar %lld | pass2+store %lld\n", e[3] - r[3], e[0] - e[3], e[1] - e[0], e[2] - e[1], r[4] - e[2]);
      }
    }
  }
  return 0;
}

void tc_destroy(CldHandle* h) {
  if (h->tc) { delete st_of(h)->itab; delete st_of(h); h->tc = nullptr; }
}

}  // namespace cld
