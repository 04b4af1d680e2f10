// flan_b200/csrc/pv_fx.h -- host-visible launch interface of pv_fx.cu (expression Functions).
#pragma once

#include <cuda_runtime.h>
#include "pv_fx.cuh"

namespace pvfx {

// The grid sampler: `total` values of the view the program's dependence selects (include/flan_b200.h, flan_b200_fx_sample).
cudaError_t launch_fx_sample( const Program & p, int64_t total, int B, bool uses_t, bool uses_f, float time_step, float bin_width,
                              float * out, int sms, cudaStream_t st );
// The program at every MF of pv (float2 [C][F][B], total = C * F * B values).
cudaError_t launch_fx_at_pv( const Program & p, const float * pv, int64_t total, int64_t F, int B, float frame_rate, float * out,
                             int sms, cudaStream_t st );

} // namespace pvfx
