// bf16 tcgen05 denoiser path (unet_tc.cu): interface used by cld_api.cu.
#pragma once
#include "common.cuh"

namespace cld {
// packs the bf16 weight images from the state-dict tensors `p` (indices of h->unet_layout)
int tc_finalize(CldHandle* h, const float* const* p, cudaStream_t s);
int tc_unet_forward(CldHandle* h, const float* x, const float* cond, const int64_t* t, float* eps, int R,
                    cudaStream_t s);
// same, with h->tbias (cond part) and h->tvec (time part) already computed by unet_cond_bias / unet_time_vec
// (tvec == nullptr: h->tvec; otherwise one row of h->tvec_all)
int tc_unet_forward_prepared(CldHandle* h, const float* x, float* eps, int R, cudaStream_t s, const float* tvec = nullptr);
void tc_destroy(CldHandle* h);
}  // namespace cld
