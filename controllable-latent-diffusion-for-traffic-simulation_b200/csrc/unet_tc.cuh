// bf16 tcgen05 denoiser path (unet_tc.cu): interface used by cld_api.cu.
#pragma once
#include "common.cuh"

namespace cld {
// slot layout of one denoiser level in the megakernel's shared-memory arena: T slots (per lane in split-time mode) in `npanels`
// 64-channel panels of `pitch` bytes, the second region at `offB`; `n_tiles` 16-slot tiles, tile i covering slots
// [slot0 + lo, slot0 + hi) (the last tile of a level that is not a multiple of 16 starts early and skips the `lo` slots it overlaps)
struct TcLevel { int T, pitch, offB, npanels, n_tiles, slot0[4], lo[4], hi[4]; };
// fills L[0..2] for `horizon` (split-time mode above 56 steps); false when the bf16 path cannot run this horizon.  The one
// owner of the bf16 horizon rule: cld_create refuses exactly the horizons for which this fails.
bool tc_level_layout(int horizon, TcLevel L[3]);
// packs the bf16 weight images from the state-dict tensors `p` (indices of h->unet_layout)
int tc_finalize(CldHandle* h, const float* const* p, cudaStream_t s);
int tc_unet_forward(CldHandle* h, const float* x, const float* cond, const int64_t* t, float* eps, int R,
                    cudaStream_t s);
// same, with h->tbias (cond part) and h->tvec (time part) already computed by unet_cond_bias / unet_time_vec
// (tvec == nullptr: h->tvec; otherwise one row of h->tvec_all)
int tc_unet_forward_prepared(CldHandle* h, const float* x, float* eps, int R, cudaStream_t s, const float* tvec = nullptr);
void tc_destroy(CldHandle* h);
}  // namespace cld
