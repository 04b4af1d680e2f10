// flan_b200/csrc/pv_modify.h -- host-visible launch interface of pv_modify.cu (PV-domain kernels).
#pragma once

#include <cuda_runtime.h>
#include "pv_modify_body.cuh"

namespace pvm {

// Result of the time-map reduction, device memory: key = float_key( maximum ), descends != 0 when some column descends.
struct MapCheck { unsigned int max_key; int descends; };

cudaError_t launch_bin_prefix( const Table & factor, int64_t rows, int B, float sample_rate, float dft, float * out, cudaStream_t st );
cudaError_t launch_frame_prefix( const Table & factor, int64_t F, int cols, float rate, float * raw_scratch, float * out, int sms, cudaStream_t st );
// Constant factor (strides (0,0)): closed-form running sum. scratch: constant_prefix_scratch_bytes() of device memory.
inline size_t constant_prefix_scratch_bytes() { return sizeof( PrefixSeg ) * PREFIX_MAX_SEGS + 256; }
cudaError_t launch_constant_prefix( const float * factor, int64_t F, float rate, void * scratch, float * out, int sms, cudaStream_t st );
cudaError_t launch_map_check( const Table & mod, int64_t F, int cols, MapCheck * check, int sms, cudaStream_t st );
// skip_if (may be null): device flag; the general row kernel returns at once when it is non-zero (the plan is valid and
// the gather kernel does the rows), the gather kernel when it is zero.
cudaError_t launch_repitch( const RepitchArgs & a, int64_t rows, const int * skip_if, cudaStream_t st );
bool repitch_shared_supported( int B );
cudaError_t launch_repitch_plan( const float * hz, int B, float bin_width, int interp, const RepitchPlan & plan, cudaStream_t st );
cudaError_t launch_repitch_shared( const RepitchArgs & a, const RepitchPlan & plan, const float * hz, int64_t rows, int sms, cudaStream_t st );
// Bin-shared time map: plan (src preset, xpos, mix) + the gather by output segments of summ.seg_len frames. With
// summ.seg_out set the kernel also leaves the phase summaries of its output rows (what pv_phase_seg_kernel would compute).
struct StretchSummary
	{
	int seg_len; int segs_per_channel;      // output frames per thread, ceil( out_frames / seg_len )
	pvk::PhaseSeg * seg_out;                // [C][segs_per_channel][B] or null
	int * nan_flag;
	pvk::PvConsts k; double P, rcpP;
	};
cudaError_t launch_stretch_planned( const StretchArgs & a, const StretchPlan & plan, const StretchSummary & summ, int C, cudaStream_t st );
// ... and its two halves, for output shards (pv_capi_multi.cu): the plan of the whole signal, then the segments
// a.seg0 .. a.seg0 + summ.segs_per_channel - 1 from the row windows that StretchArgs describes.
cudaError_t launch_stretch_plan( const StretchArgs & a, const StretchPlan & plan, cudaStream_t st );
cudaError_t launch_stretch_segments( const StretchArgs & a, const StretchPlan & plan, const StretchSummary & summ, int C, cudaStream_t st );
// Output shards [xb[i], xb[i+1]) -> rows[2i], rows[2i+1]: the input rows each one reads (stretch_window), device memory.
struct StretchWindows { static constexpr int MAX = 16; int n; int64_t xb[MAX + 1]; };
cudaError_t launch_stretch_windows( const StretchPlan & plan, int64_t F, const StretchWindows & w, int64_t * rows, cudaStream_t st );
cudaError_t launch_stretch_parallel( const StretchArgs & a, int C, cudaStream_t st );
cudaError_t launch_stretch_sequential( const StretchArgs & a, int C, cudaStream_t st );

} // namespace pvm
