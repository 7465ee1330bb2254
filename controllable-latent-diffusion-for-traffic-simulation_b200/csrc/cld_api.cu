// C ABI of libcld_b200.so (see include/cld_b200.h): handle, weight packing, dispatch, sampler loop.
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "unet_tc.cuh"

static std::string g_create_err;

namespace cld {

int fail(CldHandle* h, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (h) h->err = buf; else g_create_err = buf;
  return code;
}

int prof_begin(CldHandle* h, int kind, cudaStream_t s) {
  if (!h->profiling) return 0;
  if (h->ev_used + 2 > h->ev_pool.size()) {
    for (int i = 0; i < 64; ++i) {
      cudaEvent_t e;
      CLD_CUDA_OK(h, cudaEventCreate(&e));
      h->ev_pool.push_back(e);
    }
  }
  h->ev_kind.resize(h->ev_pool.size() / 2);
  h->ev_kind[h->ev_used / 2] = kind;
  CLD_CUDA_OK(h, cudaEventRecord(h->ev_pool[h->ev_used], s));
  return 0;
}
int prof_end(CldHandle* h, cudaStream_t s) {
  if (!h->profiling) return 0;
  CLD_CUDA_OK(h, cudaEventRecord(h->ev_pool[h->ev_used + 1], s));
  h->ev_used += 2;
  return 0;
}

template <typename T>
static int dev_alloc(CldHandle* h, T** p, size_t n) {
  if (*p) return 0;      // re-load of the decoder weights: sizes are fixed by the config, reuse
  void* q = nullptr;
  CLD_CUDA_OK(h, cudaMalloc(&q, (n ? n : 1) * sizeof(T)));
  h->allocs.push_back(q);
  *p = (T*)q;
  return 0;
}

// ---- weight pack: every pack / copy job of cld_load_unet in ONE launch (the weights change after every optimizer step)
constexpr int PACK_MAX_SRC = 160;
struct PackSrc { const float* p[PACK_MAX_SRC]; };
constexpr int PACK_BLOCK_ELEMS = 2048;
__global__ void __launch_bounds__(256) repack_all_kernel(const PackJob* __restrict__ jobs, int njobs, PackSrc src) {
  int lo = 0, hi = njobs - 1;                       // last job whose first block is <= blockIdx.x
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (jobs[mid].blk0 <= (int)blockIdx.x) lo = mid; else hi = mid - 1;
  }
  const PackJob j = jobs[lo];
  const float* __restrict__ s = src.p[j.src];
  const int base = ((int)blockIdx.x - j.blk0) * PACK_BLOCK_ELEMS;
  for (int idx = base + threadIdx.x; idx < min(j.total, base + PACK_BLOCK_ELEMS); idx += 256) {
    if (j.kind == 2) { j.dst[idx] = s[idx]; continue; }
    if (j.kind == 0) {
      const int co = idx % j.cout, ci = (idx / j.cout) % j.cin, tap = idx / (j.cout * j.cin);
      const int k = j.ks[tap];
      const float v = j.transposed ? s[((size_t)ci * j.cout + co) * j.K + k] : s[((size_t)co * j.cin + ci) * j.K + k];
      j.dst[((size_t)tap * j.cin + ci) * j.ld + j.off + co] = v;
    } else {
      const int ci = idx % j.cin, co = (idx / j.cin) % j.cout, tap = idx / (j.cout * j.cin);
      j.dst[idx] = j.transposed ? s[((size_t)ci * j.cout + co) * j.K + j.ks[tap]] : s[((size_t)co * j.cin + ci) * j.K + j.ks[tap]];
    }
  }
}

__global__ void transpose_kernel(const float* __restrict__ src, float* __restrict__ dst, int rows, int cols) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * cols) return;
  int r = idx / cols, c = idx % cols;
  dst[(size_t)c * rows + r] = src[idx];
}

__global__ void add_vec_kernel(const float* a, const float* b, float* o, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) o[i] = a[i] + b[i];
}

static int copy_vec(CldHandle* h, float** dst, const float* src, size_t n, cudaStream_t s) {
  int rc = dev_alloc(h, dst, n);
  if (rc) return rc;
  CLD_CUDA_OK(h, cudaMemcpyAsync(*dst, src, n * sizeof(float), cudaMemcpyDeviceToDevice, s));
  return 0;
}

// Channels of the residual blocks in execution order (downs.{0,1,2}.{0,1}, mid_block1, mid_block2, ups.{0,1}.{0,1}) and their slices of
// the concatenated time-bias, in the same order.
static void unet_blocks(UnetW& u, const CldConfig& c) {
  const int D = c.latent_dim, d0 = c.dims[0], d1 = c.dims[1], d2 = c.dims[2];
  const int in_ch[12] = {D, d0, d0, d1, d1, d2, d2, d2, 2 * d2, d1, 2 * d1, d0};
  const int out_ch[12] = {d0, d0, d1, d1, d2, d2, d2, d2, d1, d1, d0, d0};
  for (int e = 0; e < 12; ++e) {
    u.rb[e].cin = in_ch[e]; u.rb[e].cout = out_ch[e]; u.rb[e].tb_off = u.tb_total;
    u.tb_total += out_ch[e];
  }
}

// The denoiser's state-dict layout (DmModel.model.state_dict(), temporal.py:49-120), its packed fp32 buffers and the pack table that
// fills them from the state-dict tensors: one walk over the module tree in state-dict order (after unet_blocks).  Depends on the
// config only.
static int unet_setup(CldHandle* h) {
  const CldConfig& c = h->cfg;
  const int d = c.base_dim, D = c.latent_dim, tdim = c.base_dim + c.cond_dim;
  const int d0 = c.dims[0], d1 = c.dims[1];
  UnetW& u = h->unet;
  UnetLayout& L = h->unet_layout;
  const int k5[5] = {0, 1, 2, 3, 4}, k3[5] = {0, 1, 2, 0, 0}, k1[5] = {0, 0, 0, 0, 0};
  const int kte[5] = {1, 3, 0, 0, 0}, kto[5] = {0, 2, 0, 0, 0};   // transposed conv: taps of the even / odd output phase
  std::vector<PackJob> jobs;
  int rc = 0;
  auto buf = [&](float** p, size_t n) { if (!rc) rc = dev_alloc(h, p, n); return *p; };
  auto take = [&](int64_t numel) { L.numel.push_back(numel); return (int)L.numel.size() - 1; };
  auto job = [&](int kind, int src, float* dst, int total) -> PackJob& {
    PackJob j = {};
    j.kind = kind; j.src = src; j.dst = dst; j.total = total;
    jobs.push_back(j);
    return jobs.back();
  };
  auto vec = [&](float** dst, int n) { const int i = take(n); job(2, i, buf(dst, n), n); return i; };
  // weight `src` [cout][cin][K] (transposed: [cin][cout][K]), taps ks: -> w [tap][cin][cout] and wt [tap][cout][cin]
  auto pack = [&](ConvW& w, int src, int cout, int cin, int K, int ntaps, const int* ks, int transposed) {
    w.cin = cin; w.cout = cout; w.ntaps = ntaps;
    for (int kind = 0; kind < 2; ++kind) {
      PackJob& j = job(kind, src, buf(kind ? &w.wt : &w.w, (size_t)ntaps * cin * cout), ntaps * cin * cout);
      j.cout = cout; j.cin = cin; j.K = K; j.ntaps = ntaps; j.ld = kind ? 0 : cout; j.transposed = transposed;
      for (int t = 0; t < ntaps; ++t) j.ks[t] = ks[t];
    }
  };
  auto conv = [&](ConvW& w, int cout, int cin, int K, const int* ks, int& iw, int& ib) {
    iw = take((int64_t)cout * cin * K);
    ib = take(cout);
    pack(w, iw, cout, cin, K, K, ks, 0);
    job(2, ib, buf(&w.b, cout), cout);
  };
  auto block = [&](int e) {
    ResBlockW& rb = u.rb[e];
    BlkIdx& b = L.blk[e];
    b.tw = take((int64_t)rb.cout * tdim);
    b.tb = take(rb.cout);
    PackJob& j = job(0, b.tw, u.tb_w, rb.cout * tdim);    // time / cond projection: columns tb_off .. tb_off + cout of [tdim][tb_total]
    j.cout = rb.cout; j.cin = tdim; j.K = 1; j.ntaps = 1; j.ld = u.tb_total; j.off = rb.tb_off;
    job(2, b.tb, u.tb_b + rb.tb_off, rb.cout);
    // torch's Linear weight [cout][tdim] IS the [N][K] plane the tensor-core training forward reads: rows tb_off .. tb_off + cout
    job(2, b.tw, u.tb_wt + (size_t)rb.tb_off * tdim, rb.cout * tdim);
    conv(rb.c0, rb.cout, rb.cin, 5, k5, b.c0w, b.c0b);
    b.g0 = vec(&rb.n0.g, rb.cout);
    b.b0 = vec(&rb.n0.b, rb.cout);
    conv(rb.c1, rb.cout, rb.cout, 5, k5, b.c1w, b.c1b);
    b.g1 = vec(&rb.n1.g, rb.cout);
    b.b1 = vec(&rb.n1.b, rb.cout);
    b.rw = b.rb = -1;
    if (rb.cin != rb.cout) conv(rb.res, rb.cout, rb.cin, 1, k1, b.rw, b.rb);
  };
  L.tmlp[0] = vec(&u.t1_w, 4 * d * d);
  L.tmlp[1] = vec(&u.t1_b, 4 * d);
  L.tmlp[2] = vec(&u.t2_w, 4 * d * d);
  L.tmlp[3] = vec(&u.t2_b, d);
  {
    // SinusoidalPosEmb frequencies, same fp32 op order as the reference (diffuser_helpers.py:27-29)
    std::vector<float> f(d / 2);
    double emb = log(10000.0) / (double)(d / 2 - 1);
    for (int i = 0; i < d / 2; ++i) f[i] = expf((float)i * (float)(-emb));
    if (buf(&u.freqs, d / 2)) CLD_CUDA_OK(h, cudaMemcpy(u.freqs, f.data(), f.size() * sizeof(float), cudaMemcpyHostToDevice));
  }
  buf(&u.tb_w, (size_t)tdim * u.tb_total);
  buf(&u.tb_b, u.tb_total);
  buf(&u.tb_wt, (size_t)tdim * u.tb_total);
  for (int lvl = 0; lvl < 3; ++lvl) {             // downs.lvl: two blocks, then Downsample1d (not on the last level)
    block(2 * lvl);
    block(2 * lvl + 1);
    if (lvl < 2) conv(u.down[lvl], c.dims[lvl], c.dims[lvl], 3, k3, L.down[lvl][0], L.down[lvl][1]);
  }
  for (int lvl = 0; lvl < 2; ++lvl) {             // ups.lvl: two blocks, then Upsample1d (ConvTranspose1d k4 s2 p1)
    block(8 + 2 * lvl);
    block(9 + 2 * lvl);
    const int ch = lvl == 0 ? d1 : d0;
    const int iw = L.up[lvl][0] = take((int64_t)ch * ch * 4), ib = L.up[lvl][1] = take(ch);
    pack(u.up[lvl][0], iw, ch, ch, 4, 2, kte, 1);
    pack(u.up[lvl][1], iw, ch, ch, 4, 2, kto, 1);
    job(2, ib, buf(&u.up_b[lvl], ch), ch);
  }
  block(6);                                       // mid_block1, mid_block2
  block(7);
  conv(u.fin0, d0, d0, 5, k5, L.fin[0], L.fin[1]);   // final_conv: Conv1dBlock(d0, d0, 5), Conv1d(d0, D, 1)
  L.fin[2] = vec(&u.fin0n.g, d0);
  L.fin[3] = vec(&u.fin0n.b, d0);
  conv(u.fin1, D, d0, 1, k1, L.fin[4], L.fin[5]);
  if (rc) return rc;
  if (L.numel.size() > (size_t)PACK_MAX_SRC)
    return fail(h, CLD_ERR_UNSUPPORTED, "the denoiser has %zu tensors, the weight pack takes at most %d", L.numel.size(), PACK_MAX_SRC);
  for (PackJob& j : jobs) {
    j.blk0 = h->pack_blocks;
    h->pack_blocks += (j.total + PACK_BLOCK_ELEMS - 1) / PACK_BLOCK_ELEMS;
  }
  h->pack_njobs = (int)jobs.size();
  if ((rc = dev_alloc(h, &h->pack_jobs, jobs.size()))) return rc;
  CLD_CUDA_OK(h, cudaMemcpy(h->pack_jobs, jobs.data(), jobs.size() * sizeof(PackJob), cudaMemcpyHostToDevice));
  CLD_CUDA_OK(h, cudaStreamSynchronize(cudaStreamLegacy));   // pageable uploads: complete before any stream of the caller reads them
  return 0;
}

int check_scene(CldHandle* h, const CldScene* sc, int R) {
  const int S = sc->num_scenes, N = sc->num_samp;
  if (S < 1 || N < 1) return fail(h, CLD_ERR_ARG, "num_scenes=%d and num_samp=%d must be >= 1", S, N);
  if (!sc->scene_start && !sc->scene_start_host) {
    const int A = sc->agents_per_scene;
    if (A < 1) return fail(h, CLD_ERR_ARG, "agents_per_scene must be >= 1");
    if ((int64_t)S * A * N != R) return fail(h, CLD_ERR_ARG, "R=%d != S*A*N = %d*%d*%d", R, S, A, N);
    return 0;
  }
  if (!sc->scene_start || !sc->scene_start_host)
    return fail(h, CLD_ERR_ARG, "ragged scenes need the offsets twice: scene_start (device) and scene_start_host (host), one is NULL");
  const int32_t* o = sc->scene_start_host;
  if (o[0] != 0) return fail(h, CLD_ERR_ARG, "scene_start[0]=%d, must be 0", o[0]);
  for (int s = 0; s < S; ++s)
    if (o[s + 1] <= o[s])
      return fail(h, CLD_ERR_ARG, "scene_start must ascend: scene %d holds %d agents (scene_start[%d]=%d, [%d]=%d), every scene needs >= 1",
                  s, o[s + 1] - o[s], s, o[s], s + 1, o[s + 1]);
  if ((int64_t)o[S] * N != R) return fail(h, CLD_ERR_ARG, "scene_start[S]*N = %d*%d != R=%d", o[S], N, R);
  return 0;
}

}  // namespace cld

using namespace cld;

extern "C" {

int cld_version(void) { return 100; }

const char* cld_last_error(const CldHandle* h) { return h ? h->err.c_str() : g_create_err.c_str(); }

int cld_create(const CldConfig* cfg, CldHandle** out) {
  if (!cfg || !out) return fail(nullptr, CLD_ERR_ARG, "null argument");
  *out = nullptr;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return fail(nullptr, CLD_ERR_CUDA, "cudaGetDevice: %s", cudaGetErrorString(e));
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, dev);
  if (e != cudaSuccess) return fail(nullptr, CLD_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
  if (prop.major != 10)
    return fail(nullptr, CLD_ERR_ARCH, "libcld_b200 requires an sm_100 (B200) device, found sm_%d%d; there is no fallback",
                prop.major, prop.minor);
  if (cfg->horizon % 4 || cfg->horizon < 8 || cfg->horizon > CLD_MAX_T)
    return fail(nullptr, CLD_ERR_ARG, "horizon must be a multiple of 4 in [8,%d]", CLD_MAX_T);
  if (cfg->latent_dim != 4) return fail(nullptr, CLD_ERR_UNSUPPORTED, "latent_dim must be 4");
  if (cfg->base_dim < 2 || cfg->base_dim > 64 || cfg->base_dim % 4)
    return fail(nullptr, CLD_ERR_UNSUPPORTED, "base_dim must be a multiple of 4 in [4,64]");
  for (int i = 0; i < 3; ++i)
    if (cfg->dims[i] % 8 || cfg->dims[i] < 8) return fail(nullptr, CLD_ERR_UNSUPPORTED, "dims must be multiples of 8");
  if (cfg->cond_dim % 4 || cfg->cond_dim < 4) return fail(nullptr, CLD_ERR_UNSUPPORTED, "cond_dim must be a multiple of 4");
  if (cfg->max_rows < 1) return fail(nullptr, CLD_ERR_ARG, "max_rows must be positive");
  if (cfg->n_timesteps < 1) return fail(nullptr, CLD_ERR_ARG, "n_timesteps must be positive");
  {
    TcLevel levels[3];
    const bool t_ok = tc_level_layout(cfg->horizon, levels);      // the horizons tc_finalize can lay out, no others
    if (cfg->precision == CLD_PREC_BF16 && !(cfg->dims[0] == 64 && cfg->dims[1] == 128 && cfg->dims[2] == 256 && t_ok && cfg->hidden == 64))
      return fail(nullptr, CLD_ERR_UNSUPPORTED,
                  "the bf16 tensor-core path is built for dims (64,128,256), hidden 64 and a horizon of 16..56 (8 rows per CTA) or 64..104 in "
                  "multiples of 8 (4 rows per CTA as two half-horizon lanes); use precision fp32 for this configuration");
  }
  CldHandle* h = new CldHandle();
  h->cfg = *cfg;
  h->device = dev;
  h->num_sms = prop.multiProcessorCount;
  // bf16-precision mode runs the LSTM decoder (forward and BPTT) on the tensor pipe; CLD_LSTM_SIMT=1 keeps the fp32 SIMT kernels
  h->use_lstm_tc = cfg->precision == CLD_PREC_BF16 && cfg->hidden == 64 && getenv("CLD_LSTM_SIMT") == nullptr;
  h->env_lstm_bwd_simt = getenv("CLD_LSTM_BWD_SIMT") != nullptr;
  h->env_guidance_nofork = getenv("CLD_GUIDANCE_NOFORK") != nullptr;
  h->env_lstm_prof = getenv("CLD_LSTM_PROF") != nullptr;
  h->env_map_stats = getenv("CLD_MAP_STATS") != nullptr;
  h->env_map_exhaustive = getenv("CLD_MAP_EXHAUSTIVE") != nullptr;
  h->env_train_serial = getenv("CLD_TRAIN_SERIAL") != nullptr;
  if (const char* e = getenv("CLD_LSTM_PF")) h->env_lstm_pf = atoi(e);
  const int T = cfg->horizon;
  const size_t MR = cfg->max_rows;
  size_t ae = (size_t)T * cfg->dims[0];
  if ((size_t)(T / 2) * cfg->dims[1] > ae) ae = (size_t)(T / 2) * cfg->dims[1];
  if ((size_t)(T / 4) * cfg->dims[2] > ae) ae = (size_t)(T / 4) * cfg->dims[2];
  h->act_elems = ae;
  unet_blocks(h->unet, *cfg);
  const int tb_total = h->unet.tb_total;
  int rc = 0;
  for (int i = 0; i < 7 && !rc; ++i) rc = dev_alloc(h, &h->act[i], MR * ae);
  if (!rc) rc = dev_alloc(h, &h->tcm, MR * (cfg->base_dim + cfg->cond_dim));
  if (!rc) rc = dev_alloc(h, &h->tbias, MR * tb_total);
  if (!rc) rc = dev_alloc(h, &h->tvec, tb_total);
  if (!rc) rc = dev_alloc(h, &h->tvec_all, (size_t)cfg->n_timesteps * tb_total);
  if (!rc) rc = dev_alloc(h, &h->stash, (size_t)2 * T * ((MR + 63) / 64 * 64) * 5 * cfg->hidden);
  if (!rc) rc = dev_alloc(h, &h->ws_act, MR * T * 2);
  if (!rc) rc = dev_alloc(h, &h->ws_h0, MR * cfg->hidden);
  if (!rc) rc = dev_alloc(h, &h->ws_dh0, (size_t)T * MR * cfg->hidden);
  if (!rc) rc = dev_alloc(h, &h->ws_traj, MR * T * 6);
  if (!rc) rc = dev_alloc(h, &h->ws_dtraj, MR * T * 4);
  if (!rc && h->use_lstm_tc) rc = dev_alloc(h, &h->ws_dtraj2, MR * T * 4);
  if (!rc) rc = dev_alloc(h, &h->ws_dacc, MR * T);
  if (!rc) rc = dev_alloc(h, &h->map_work, MR * T + 8);
  if (!rc && cudaMemset(h->map_work, 0, 8 * sizeof(int)) != cudaSuccess) rc = fail(h, CLD_ERR_CUDA, "cudaMemset of the map work list failed");
  if (!rc) rc = dev_alloc(h, &h->ws_loss, 7 * MR);
  if (!rc) rc = dev_alloc(h, &h->ws_eps, MR * T * cfg->latent_dim);
  if (!rc) rc = dev_alloc(h, &h->ws_mean, MR * T * cfg->latent_dim);
  if (!rc) rc = dev_alloc(h, &h->ws_x, MR * T * cfg->latent_dim);
  if (!rc) rc = dev_alloc(h, &h->ws_t, MR);
  if (!rc) rc = unet_setup(h);
  if (rc) {
    g_create_err = h->err;
    cld_destroy(h);
    return rc;
  }
  *out = h;
  return CLD_OK;
}

void cld_destroy(CldHandle* h) {
  if (!h) return;
  tc_destroy(h);
  lstm_tc_destroy(h);
  train_destroy(h);
  train_tc_destroy(h);
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h->ev_join) cudaEventDestroy(h->ev_join);
  if (h->ev_tvec) cudaEventDestroy(h->ev_tvec);
  if (h->aux_stream) cudaStreamDestroy(h->aux_stream);
  for (cudaEvent_t e : h->ev_pool) cudaEventDestroy(e);
  for (void* p : h->allocs) cudaFree(p);
  delete h;
}

int cld_load_unet(CldHandle* h, const float* const* p, const int64_t* numels, int n, void* stream) {
  if (!h || !p) return fail(h, CLD_ERR_ARG, "null argument");
  const UnetLayout& L = h->unet_layout;
  if (n != (int)L.numel.size()) return fail(h, CLD_ERR_ARG, "cld_load_unet: expected %zu tensors, got %d", L.numel.size(), n);
  PackSrc src;
  for (int i = 0; i < n; ++i) {
    if (!p[i]) return fail(h, CLD_ERR_ARG, "cld_load_unet: tensor %d is null", i);
    if (numels && numels[i] != L.numel[i])
      return fail(h, CLD_ERR_ARG, "cld_load_unet: tensor %d has %lld elements, expected %lld", i, (long long)numels[i], (long long)L.numel[i]);
    src.p[i] = p[i];
  }
  cudaStream_t s = (cudaStream_t)stream;
  repack_all_kernel<<<h->pack_blocks, 256, 0, s>>>(h->pack_jobs, h->pack_njobs, src);
  CLD_LAUNCH_OK(h, "repack_all_kernel");
  h->tvec_all_valid = false;
  train_invalidate(h);
  int rc;
  if (h->cfg.precision == CLD_PREC_BF16 && (rc = tc_finalize(h, p, s))) return rc;
  h->unet.loaded = true;
  return CLD_OK;
}

int cld_load_decoder(CldHandle* h, const float* const* p, int n, void* stream) {
  if (!h || !p) return fail(h, CLD_ERR_ARG, "null argument");
  if (n != 12) return fail(h, CLD_ERR_ARG, "cld_load_decoder: expected 12 tensors, got %d", n);
  cudaStream_t s = (cudaStream_t)stream;
  const int H = h->cfg.hidden, G = 4 * H, C = h->cfg.cond_dim, D = h->cfg.latent_dim;
  DecoderW& w = h->dec;
  int rc;
  auto transposed = [&](float** dst, const float* src, int rows, int cols) -> int {
    int r = dev_alloc(h, dst, (size_t)rows * cols);
    if (r) return r;
    transpose_kernel<<<(rows * cols + 255) / 256, 256, 0, s>>>(src, *dst, rows, cols);
    CLD_LAUNCH_OK(h, "transpose_kernel");
    return 0;
  };
  if ((rc = transposed(&w.wih0, p[0], G, D))) return rc;
  if ((rc = transposed(&w.whh0, p[1], G, H))) return rc;
  if ((rc = transposed(&w.wih1, p[4], G, H))) return rc;
  if ((rc = transposed(&w.whh1, p[5], G, H))) return rc;
  if ((rc = copy_vec(h, &w.wih0_raw, p[0], (size_t)G * D, s))) return rc;
  if ((rc = copy_vec(h, &w.whh0_raw, p[1], (size_t)G * H, s))) return rc;
  if ((rc = copy_vec(h, &w.wih1_raw, p[4], (size_t)G * H, s))) return rc;
  if ((rc = copy_vec(h, &w.whh1_raw, p[5], (size_t)G * H, s))) return rc;
  if ((rc = dev_alloc(h, &w.b0, G))) return rc;
  if ((rc = dev_alloc(h, &w.b1, G))) return rc;
  add_vec_kernel<<<(G + 255) / 256, 256, 0, s>>>(p[2], p[3], w.b0, G);
  add_vec_kernel<<<(G + 255) / 256, 256, 0, s>>>(p[6], p[7], w.b1, G);
  CLD_LAUNCH_OK(h, "add_vec_kernel");
  if ((rc = transposed(&w.c2h_w, p[8], H, C))) return rc;
  if ((rc = copy_vec(h, &w.c2h_b, p[9], H, s))) return rc;
  if ((rc = copy_vec(h, &w.h2a_w, p[10], 2 * H, s))) return rc;
  if ((rc = copy_vec(h, &w.h2a_b, p[11], 2, s))) return rc;
  CLD_CUDA_OK(h, cudaStreamSynchronize(s));
  w.loaded = true;
  return CLD_OK;
}

int cld_set_schedule(CldHandle* h, const float* x_t_cof, const float* noise_cof, const float* logvar,
                     const float* sqrt_recip, const float* sqrt_recipm1, const float* sqrt_acp,
                     const float* sqrt_1macp, int n) {
  if (!h || !x_t_cof || !noise_cof || !logvar) return fail(h, CLD_ERR_ARG, "null argument");
  if (n != h->cfg.n_timesteps) return fail(h, CLD_ERR_ARG, "schedule length %d != n_timesteps %d", n, h->cfg.n_timesteps);
  Schedule& sc = h->sched;
  sc.x_t_cof.assign(x_t_cof, x_t_cof + n);
  sc.noise_cof.assign(noise_cof, noise_cof + n);
  sc.logvar.assign(logvar, logvar + n);
  auto opt = [&](std::vector<float>& v, const float* p) { if (p) v.assign(p, p + n); else v.assign(n, 0.f); };
  opt(sc.sqrt_recip, sqrt_recip); opt(sc.sqrt_recipm1, sqrt_recipm1); opt(sc.sqrt_acp, sqrt_acp); opt(sc.sqrt_1macp, sqrt_1macp);
  sc.loaded = true;
  ++h->sched_version;
  return CLD_OK;
}

static int check_rows(CldHandle* h, int R) {
  if (!h) return CLD_ERR_ARG;
  if (R < 1 || R > h->cfg.max_rows) return fail(h, CLD_ERR_ARG, "R=%d outside [1, max_rows=%d]", R, h->cfg.max_rows);
  return 0;
}

static int unet_dispatch(CldHandle* h, const float* x, const float* cond, const int64_t* t, float* eps, int R,
                         cudaStream_t s) {
  if (!h->unet.loaded) return fail(h, CLD_ERR_STATE, "denoiser weights not loaded");
  if (h->cfg.precision == CLD_PREC_BF16) return tc_unet_forward(h, x, cond, t, eps, R, s);
  return unet_forward_fp32(h, x, cond, t, eps, R, s);
}

int cld_unet_forward(CldHandle* h, const float* x, const float* cond, const int64_t* t, float* eps_out, int R,
                     void* stream) {
  int rc = check_rows(h, R);
  if (rc) return rc;
  if (!x || !cond || !t || !eps_out) return fail(h, CLD_ERR_ARG, "null argument");
  return unet_dispatch(h, x, cond, t, eps_out, R, (cudaStream_t)stream);
}

/* ---- SURVEY.md sec. 8 f-2: denoiser training step (PPO update / DM loss) ---- */
int cld_unet_train_forward(CldHandle* h, const float* x, const float* cond, const int64_t* t, float* eps_out, int R, void* stream) {
  int rc = check_rows(h, R);
  if (rc) return rc;
  if (!x || !cond || !t || !eps_out) return fail(h, CLD_ERR_ARG, "null argument");
  if (!h->unet.loaded) return fail(h, CLD_ERR_STATE, "denoiser weights not loaded");
  return unet_train_forward(h, x, cond, t, eps_out, R, (cudaStream_t)stream);
}

int cld_unet_backward(CldHandle* h, const float* d_eps, float* const* grads, int n, float* dx_out, int R, void* stream) {
  int rc = check_rows(h, R);
  if (rc) return rc;
  if (!d_eps || !grads) return fail(h, CLD_ERR_ARG, "null argument");
  for (int i = 0; i < n; ++i)
    if (!grads[i]) return fail(h, CLD_ERR_ARG, "gradient pointer %d is null", i);
  return unet_train_backward(h, d_eps, grads, n, dx_out, R, (cudaStream_t)stream);
}

int cld_ppo_head(CldHandle* h, const float* eps, const float* x_t, const float* x_tm1, const int64_t* t, const float* logp_old,
                 const float* reward, float baseline, const float* baseline_dev, float clip_eps, float* logp_new_out, float* loss_out,
                 float* d_eps_out, int R, void* stream) {
  int rc = check_rows(h, R);
  if (rc) return rc;
  if (!eps || !x_t || !x_tm1 || !t || !logp_old || !reward) return fail(h, CLD_ERR_ARG, "null argument");
  return ppo_head(h, eps, x_t, x_tm1, t, logp_old, reward, baseline, baseline_dev, clip_eps, logp_new_out, loss_out, d_eps_out, R,
                  (cudaStream_t)stream);
}

int cld_mse_head(CldHandle* h, const float* eps, const float* noise, float* loss_out, float* d_eps_out, int R, void* stream) {
  int rc = check_rows(h, R);
  if (rc) return rc;
  if (!eps || !noise) return fail(h, CLD_ERR_ARG, "null argument");
  return mse_head(h, eps, noise, loss_out, d_eps_out, R, (cudaStream_t)stream);
}

int cld_ppo_grad(CldHandle* h, const float* x_t, const float* x_tm1, const float* cond, const int64_t* t, const float* logp_old,
                 const float* reward, float baseline, const float* baseline_dev, float clip_eps, float* const* grads, int n,
                 float* logp_new_out, float* loss_out, int R, void* stream) {
  int rc = check_rows(h, R);
  if (rc) return rc;
  if (!x_t || !x_tm1 || !cond || !t || !logp_old || !reward || !grads) return fail(h, CLD_ERR_ARG, "null argument");
  if (!h->unet.loaded) return fail(h, CLD_ERR_STATE, "denoiser weights not loaded");
  cudaStream_t s = (cudaStream_t)stream;
  if ((rc = unet_train_forward(h, x_t, cond, t, h->ws_eps, R, s))) return rc;
  float* d_eps = train_deps_buffer(h);
  if ((rc = ppo_head(h, h->ws_eps, x_t, x_tm1, t, logp_old, reward, baseline, baseline_dev, clip_eps, logp_new_out, loss_out, d_eps, R, s)))
    return rc;
  for (int i = 0; i < n; ++i)
    if (!grads[i]) return fail(h, CLD_ERR_ARG, "gradient pointer %d is null", i);
  return unet_train_backward(h, d_eps, grads, n, nullptr, R, s);
}

int cld_adam_step_dev(CldHandle* h, float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t numel, const double* lr_dev,
                      int64_t* step_dev, double beta1, double beta2, double eps, double weight_decay, void* stream) {
  if (!h || !params || !grads || !exp_avg || !exp_avg_sq || !lr_dev || !step_dev) return fail(h, CLD_ERR_ARG, "null argument");
  if (numel < 1) return fail(h, CLD_ERR_ARG, "numel must be positive");
  return adam_step_dev(h, params, grads, exp_avg, exp_avg_sq, (size_t)numel, lr_dev, (long long*)step_dev, beta1, beta2, eps, weight_decay,
                       (cudaStream_t)stream);
}

int cld_train_set_precision(CldHandle* h, int tf32) {
  if (!h) return CLD_ERR_ARG;
  h->train_tf32 = tf32 != 0;
  return CLD_OK;
}

int cld_adam_step(CldHandle* h, float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t numel, double lr,
                  double beta1, double beta2, double eps, double weight_decay, int step, void* stream) {
  if (!h || !params || !grads || !exp_avg || !exp_avg_sq) return fail(h, CLD_ERR_ARG, "null argument");
  if (numel < 1 || step < 1) return fail(h, CLD_ERR_ARG, "numel and step must be positive");
  return adam_step(h, params, grads, exp_avg, exp_avg_sq, (size_t)numel, lr, beta1, beta2, eps, weight_decay, step, (cudaStream_t)stream);
}

int cld_unet_debug_stage(CldHandle* h, int stage_index, float* out, int R, void* stream) {
  (void)R; (void)stream;
  if (!h) return CLD_ERR_ARG;
  h->dbg_stage = out ? stage_index : -1;
  h->dbg_out = out;
  return out ? unet_stage_elems(h, stage_index) : 0;
}

int cld_posterior_step(CldHandle* h, const float* x, const float* eps, const float* noise, int t, int t_next,
                       int sampler, float* x_out, float* mean_out, int R, void* stream) {
  int rc = check_rows(h, R);
  if (rc) return rc;
  if (!x || !eps) return fail(h, CLD_ERR_ARG, "null argument");
  if (!noise && x_out && sampler == CLD_SAMPLER_DDPM && t != 0)
    return fail(h, CLD_ERR_ARG, "noise tensor required for a DDPM step with t != 0");
  return posterior_step(h, x, eps, noise, 0, 0, 0, t, t_next, sampler, x_out, mean_out, R, (cudaStream_t)stream);
}

int cld_add_noise(CldHandle* h, const float* mean, const float* noise, int t, float* x_out, int R, void* stream) {
  int rc = check_rows(h, R);
  if (rc) return rc;
  if (!mean || !x_out || (!noise && t != 0)) return fail(h, CLD_ERR_ARG, "null argument");
  return add_noise(h, mean, noise, 0, 0, 0, t, x_out, R, (cudaStream_t)stream);
}

int cld_decode_rollout(CldHandle* h, const float* z, const float* cond, const float* curr, float* act_out,
                       float* traj_out, int R, void* stream) {
  int rc = check_rows(h, R);
  if (rc) return rc;
  if (!z || !cond || !curr) return fail(h, CLD_ERR_ARG, "null argument");
  return decode_rollout(h, z, cond, curr, act_out, traj_out, false, R, (cudaStream_t)stream);
}

int cld_unicycle(CldHandle* h, const float* curr, const float* u, float* state_out, int R, void* stream) {
  if (!h || !curr || !u || !state_out || R < 1) return fail(h, CLD_ERR_ARG, "bad argument");
  return unicycle(h, curr, u, state_out, R, (cudaStream_t)stream);
}

int cld_indicators(CldHandle* h, const float* traj, const CldScene* scene, uint8_t* offroad_out, float* coll_out,
                   float* reward_out, int R, void* stream) {
  if (!h || !traj || R < 1) return fail(h, CLD_ERR_ARG, "bad argument");
  int rc;
  if (scene && (rc = check_scene(h, scene, R))) return rc;
  return indicators(h, traj, scene, offroad_out, coll_out, reward_out, R, (cudaStream_t)stream);
}

// checks CldGuidanceConfig.grad_steps and, for a multi-step Adam call, allocates the moment buffers on first use
static int guidance_prepare_steps(CldHandle* h, const CldGuidanceConfig* g) {
  if (g->grad_steps < 0) return fail(h, CLD_ERR_ARG, "grad_steps must be >= 0 (0 and 1 both mean one iteration), got %d", g->grad_steps);
  if (g->grad_steps <= 1 || g->optimizer != CLD_OPT_ADAM) return 0;
  const size_t n = (size_t)h->cfg.max_rows * h->cfg.horizon * 4;
  int rc;
  if ((rc = dev_alloc(h, &h->ws_adam_m, n))) return rc;
  return dev_alloc(h, &h->ws_adam_v, n);
}

// h0 == nullptr: compute cond2hidden(cond) first; otherwise cond is unused.  g->grad_steps iterations of decode (with stash) ->
// losses -> BPTT + optimizer step: iteration 1 reads z_mean, later ones the z_out of the one before (in place: each row reads
// its z before it writes it); grad_out / loss_out keep the last iteration's values.
static int guidance_step_impl(CldHandle* h, const float* z_mean, const float* cond, const float* h0, const float* curr,
                              const CldScene* scene, const CldGuidanceConfig* g, float* z_out, float* grad_out,
                              float* loss_out, int R, cudaStream_t s) {
  int rc;
  if (!h0) {
    if ((rc = decode_h0(h, cond, h->ws_h0, R, s))) return rc;
    h0 = h->ws_h0;
  }
  // bf16 mode without per-row loss output (the sampler): the two loss kernels run concurrently, each into its own buffer
  float* dmap = (h->use_lstm_tc && !loss_out && g->w_map_collision != 0.f && !h->env_lstm_bwd_simt &&
                 !h->env_guidance_nofork) ? h->ws_dtraj2 : nullptr;
  float* dacc = g->w_acc_limit != 0.f ? h->ws_dacc : nullptr;
  const int steps = g->grad_steps > 1 ? g->grad_steps : 1;
  const bool moments = steps > 1 && g->optimizer == CLD_OPT_ADAM;
  if (moments && !h->ws_adam_m) return fail(h, CLD_ERR_STATE, "internal: Adam moment buffers not allocated");
  for (int it = 1; it <= steps; ++it) {
    const float* z = it == 1 ? z_mean : z_out;
    const bool last = it == steps;
    GuideOpt opt;
    opt.iter = it;
    if (moments) {
      // torch.optim.Adam derives its scalar factors in double: step_size = lr / bc1, bc2 ** 0.5
      opt.m = h->ws_adam_m; opt.v = h->ws_adam_v;
      opt.step_size = (float)((double)g->lr / (1.0 - pow(0.9, it)));
      opt.bc2_sqrt = (float)sqrt(1.0 - pow(0.999, it));
    }
    if ((rc = decode_rollout_h0(h, z, h0, curr, h->ws_act, h->ws_traj, true, R, s))) return rc;
    if ((rc = guidance_loss_grad(h, h->ws_traj, scene, g, h->ws_dtraj, dmap, dacc, last ? loss_out : nullptr, R, s))) return rc;
    if ((rc = decode_backward_update2(h, z, h->ws_act, curr, h->ws_dtraj, dmap, dacc, g, opt, z_out, last ? grad_out : nullptr, R, s)))
      return rc;
  }
  return 0;
}

int cld_guidance_step(CldHandle* h, const float* z_mean, const float* cond, const float* curr, const CldScene* scene,
                      const CldGuidanceConfig* g, float* z_out, float* grad_out, float* loss_out, int R, void* stream) {
  int rc = check_rows(h, R);
  if (rc) return rc;
  if (!z_mean || !cond || !curr || !scene || !g || !z_out) return fail(h, CLD_ERR_ARG, "null argument");
  if ((rc = check_scene(h, scene, R))) return rc;
  if ((rc = guidance_prepare_steps(h, g))) return rc;
  if (g->w_map_collision != 0.f && (rc = guidance_prepare_maps(h, scene, (cudaStream_t)stream))) return rc;
  return guidance_step_impl(h, z_mean, cond, nullptr, curr, scene, g, z_out, grad_out, loss_out, R, (cudaStream_t)stream);
}

int cld_sample(CldHandle* h, const float* x_init, const float* noises, uint64_t seed, int64_t row_offset, const float* cond,
               const float* curr, const CldScene* scene, const CldGuidanceConfig* g, int stride, int sampler,
               float* x0_out, float* x1_out, int* x1_valid, float* traj_out, uint8_t* offroad_out, float* coll_out,
               int R, void* stream) {
  if (!h || !cond) return fail(h, CLD_ERR_ARG, "null argument");
  if (!x_init && seed == 0) return fail(h, CLD_ERR_ARG, "either x_init or a non-zero seed (in-kernel Philox initial state) is required");
  if (row_offset < 0) return fail(h, CLD_ERR_ARG, "row_offset must be >= 0");
  if (R < 1 || stride < 1) return fail(h, CLD_ERR_ARG, "bad R / stride");
  if ((traj_out || offroad_out || coll_out || g) && !curr) return fail(h, CLD_ERR_ARG, "curr states required");
  if ((offroad_out || coll_out || g) && !scene) return fail(h, CLD_ERR_ARG, "scene tensors required");
  if (!h->sched.loaded) return fail(h, CLD_ERR_STATE, "schedule not set");
  int rc;
  if (scene && (rc = check_scene(h, scene, R))) return rc;
  if (g && (rc = guidance_prepare_steps(h, g))) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  const CldConfig& c = h->cfg;
  const int T = c.horizon, D = c.latent_dim, n_t = c.n_timesteps;
  const size_t row_e = (size_t)T * D;
  std::vector<int> steps;
  for (int i = 0; i < n_t; i += stride) steps.push_back(i);
  const int K = (int)steps.size();
  if (x1_valid) *x1_valid = 0;
  // chunks of whole scenes, packed greedily in batch order up to max_rows rows: {first scene, first row} of every chunk, then the end
  std::vector<int> chunk_scene, chunk_row;
  if (scene) {
    const int S = scene->num_scenes, N = scene->num_samp;
    auto first_agent = [&](int sidx) { return scene->scene_start ? scene->scene_start_host[sidx] : sidx * scene->agents_per_scene; };
    for (int sidx = 0; sidx < S; ++sidx) {
      const int rows = (first_agent(sidx + 1) - first_agent(sidx)) * N;
      if (rows > c.max_rows) return fail(h, CLD_ERR_ARG, "max_rows=%d is smaller than one scene (scene %d: A*N=%d)", c.max_rows, sidx, rows);
      if (chunk_scene.empty() || (first_agent(sidx + 1) - first_agent(chunk_scene.back())) * N > c.max_rows) {
        chunk_scene.push_back(sidx);
        chunk_row.push_back(first_agent(sidx) * N);
      }
    }
    chunk_scene.push_back(S);
  } else {
    for (int r0 = 0; r0 < R; r0 += c.max_rows) chunk_row.push_back(r0);
  }
  chunk_row.push_back(R);
  for (size_t ci = 0; ci + 1 < chunk_row.size(); ++ci) {
    const int r0 = chunk_row[ci], Rc = chunk_row[ci + 1] - r0;
    CldScene sub;
    const CldScene* sc = nullptr;
    if (scene) {
      sub = *scene;
      const size_t a0 = (size_t)r0 / scene->num_samp;
      sub.num_scenes = chunk_scene[ci + 1] - chunk_scene[ci];
      // a chunk's offsets keep their values: the kernels subtract scene_start_host[0], its first agent
      if (sub.scene_start) { sub.scene_start += chunk_scene[ci]; sub.scene_start_host += chunk_scene[ci]; }
      if (sub.extent) sub.extent += a0 * 3;
      if (sub.world_from_agent) sub.world_from_agent += a0 * 9;
      if (sub.raster_from_agent) sub.raster_from_agent += a0 * 9;
      if (sub.curr_speed) sub.curr_speed += a0;
      if (sub.drivable_map) sub.drivable_map += a0 * scene->map_h * (scene->map_packed ? (scene->map_w + 7) / 8 : scene->map_w);
      if (sub.target_pos) sub.target_pos += a0 * 2;
      if (sub.others_pos) sub.others_pos += a0 * scene->num_others * T * 2;
      if (sub.others_avail) sub.others_avail += a0 * scene->num_others * T;
      if (sub.target_speed) sub.target_speed += a0 * T;
      if (sub.wp_target) sub.wp_target += a0 * 2;
      if (sub.wp_mode) sub.wp_mode += a0;
      if (sub.wp_time) sub.wp_time += a0;
      if (sub.wp_dist) sub.wp_dist += a0;
      if (sub.wp_weight) sub.wp_weight += a0;
      sc = &sub;
    }
    const float* condc = cond + (size_t)r0 * c.cond_dim;
    const float* currc = curr ? curr + (size_t)r0 * 4 : nullptr;
    float* x = h->ws_x;
    // Philox counters are indexed by the GLOBAL row id (row_offset + r0 + local row): results do not depend on how rows are
    // sharded over ranks, chunked by max_rows or split into lanes (SURVEY.md sec. 8e)
    const uint64_t idx_base = ((uint64_t)row_offset + (uint64_t)r0) * (uint64_t)(row_e / 4);
    if (x_init) {
      CLD_CUDA_OK(h, cudaMemcpyAsync(x, x_init + r0 * row_e, Rc * row_e * sizeof(float), cudaMemcpyDeviceToDevice, s));
    } else if ((rc = philox_fill(h, seed, ~0ull, idx_base, x, Rc, s))) {
      return rc;
    }
    // bf16 path: the cond half of every block's time/cond projection is step-invariant -> once per chunk
    const bool split_bias = (c.precision == CLD_PREC_BF16);
    if (split_bias && (rc = unet_cond_bias(h, condc, Rc, s))) return rc;
    if (split_bias && !h->tvec_all_valid) {
      // the time part of every block's bias depends on the timestep only: one table per weight load instead of a kernel per step
      for (int t = 0; t < n_t; ++t)
        if ((rc = unet_time_vec_to(h, t, h->tvec_all + (size_t)t * h->unet.tb_total, s))) return rc;
      if (!h->ev_tvec) CLD_CUDA_OK(h, cudaEventCreateWithFlags(&h->ev_tvec, cudaEventDisableTiming));
      CLD_CUDA_OK(h, cudaEventRecord(h->ev_tvec, s));
      h->tvec_stream = s;
      h->tvec_all_valid = true;
    } else if (split_bias && s != h->tvec_stream && h->ev_tvec) {
      CLD_CUDA_OK(h, cudaStreamWaitEvent(s, h->ev_tvec, 0));
    }
    // so is the tile table that screens the map-collision term (the maps of this chunk)
    if (g && g->w_map_collision != 0.f && (rc = guidance_prepare_maps(h, sc, s))) return rc;
    // LSTM initial state (cond2hidden) is step-invariant as well
    if ((g || traj_out || offroad_out || coll_out) && (rc = decode_h0(h, condc, h->ws_h0, Rc, s))) return rc;
    for (int k = 0; k < K; ++k) {
      const int i = steps[K - 1 - k];
      const int i_next = (k + 1 < K) ? steps[K - 2 - k] : -1;
      const float* nz = noises ? noises + ((size_t)k * R + r0) * row_e : nullptr;
      if (!noises && seed == 0 && sampler == CLD_SAMPLER_DDPM && i != 0)
        return fail(h, CLD_ERR_ARG, "either a noise tensor or a non-zero seed is required");
      if ((rc = prof_begin(h, 0, s))) return rc;
      if (split_bias) {
        if ((rc = tc_unet_forward_prepared(h, x, h->ws_eps, Rc, s, h->tvec_all + (size_t)i * h->unet.tb_total))) return rc;
      } else {
        if ((rc = fill_t(h, h->ws_t, i, Rc, s))) return rc;
        if ((rc = unet_dispatch(h, x, condc, h->ws_t, h->ws_eps, Rc, s))) return rc;
      }
      if ((rc = prof_end(h, s))) return rc;
      const bool guided = (g != nullptr) && i != 0;
      const uint64_t seq = (uint64_t)k;
      if (!guided) {
        if ((rc = prof_begin(h, 1, s))) return rc;
        if ((rc = posterior_step(h, x, h->ws_eps, nz, seed, seq, idx_base, i, i_next, sampler, x, nullptr, Rc, s))) return rc;
        if ((rc = prof_end(h, s))) return rc;
      } else {
        if ((rc = prof_begin(h, 1, s))) return rc;
        if ((rc = posterior_step(h, x, h->ws_eps, nullptr, 0, 0, 0, i, i_next, sampler, nullptr, h->ws_mean, Rc, s))) return rc;
        if ((rc = prof_end(h, s))) return rc;
        if ((rc = prof_begin(h, 2, s))) return rc;
        // DDIM (eta = 0) injects no noise: the guidance update writes the next state directly
        const bool noiseless = sampler != CLD_SAMPLER_DDPM;
        if ((rc = guidance_step_impl(h, h->ws_mean, condc, h->ws_h0, currc, sc, g, noiseless ? x : h->ws_mean, nullptr, nullptr, Rc, s))) return rc;
        if ((rc = prof_end(h, s))) return rc;
        if (!noiseless) {
          if ((rc = prof_begin(h, 1, s))) return rc;
          if ((rc = add_noise(h, h->ws_mean, nz, seed, seq, idx_base, i, x, Rc, s))) return rc;
          if ((rc = prof_end(h, s))) return rc;
        }
      }
      if (i == 1 && x1_out) {
        CLD_CUDA_OK(h, cudaMemcpyAsync(x1_out + r0 * row_e, x, Rc * row_e * sizeof(float), cudaMemcpyDeviceToDevice, s));
        if (x1_valid) *x1_valid = 1;
      }
    }
    if (x0_out)
      CLD_CUDA_OK(h, cudaMemcpyAsync(x0_out + r0 * row_e, x, Rc * row_e * sizeof(float), cudaMemcpyDeviceToDevice, s));
    if (traj_out || offroad_out || coll_out) {
      float* tr = traj_out ? traj_out + (size_t)r0 * T * 6 : h->ws_traj;
      if ((rc = prof_begin(h, 3, s))) return rc;
      if ((rc = decode_rollout_h0(h, x, h->ws_h0, currc, h->ws_act, tr, false, Rc, s))) return rc;
      if (offroad_out || coll_out) {
        if ((rc = indicators(h, tr, sc, offroad_out ? offroad_out + (size_t)r0 * T : nullptr,
                             coll_out ? coll_out + r0 : nullptr, nullptr, Rc, s)))
          return rc;
      }
      if ((rc = prof_end(h, s))) return rc;
    }
  }
  return CLD_OK;
}

unsigned long long cld_launch_count(const CldHandle* h) { return h ? h->launches : 0ull; }

int cld_profile_begin(CldHandle* h) {
  if (!h) return CLD_ERR_ARG;
  h->profiling = true;
  h->ev_used = 0;
  return CLD_OK;
}

int cld_profile_end(CldHandle* h, double* ms_by_kind, int* count_by_kind, int nkinds) {
  if (!h || !ms_by_kind || !count_by_kind) return fail(h, CLD_ERR_ARG, "null argument");
  for (int k = 0; k < nkinds; ++k) { ms_by_kind[k] = 0.0; count_by_kind[k] = 0; }
  if (h->ev_used) CLD_CUDA_OK(h, cudaEventSynchronize(h->ev_pool[h->ev_used - 1]));
  for (size_t i = 0; i + 1 < h->ev_used; i += 2) {
    float ms = 0.f;
    CLD_CUDA_OK(h, cudaEventElapsedTime(&ms, h->ev_pool[i], h->ev_pool[i + 1]));
    int k = h->ev_kind[i / 2];
    if (k >= 0 && k < nkinds) { ms_by_kind[k] += ms; count_by_kind[k] += 1; }
  }
  h->profiling = false;
  h->ev_used = 0;
  return CLD_OK;
}

}  // extern "C"
