// flan_b200/csrc/pv_launch.h -- host-visible launch interface of pv_kernels.cu.
#pragma once

#include <cuda_runtime.h>
#include "pv_body.cuh"
#include "pv_policy.h"

namespace pvk {

struct PhaseSegArgs
	{
	const float2 * pv;
	int64_t pv_channel_stride;
	int64_t frame_begin, frame_end;
	int seg_len, segs_per_channel, B;
	PhaseSeg * seg_out;         // [C][segs_per_channel][B]
	int * nan_flag;             // set to 1 when a NaN/Inf magnitude or frequency is seen (AudioPV.cpp:88)
	PvConsts k;
	double P, rcpP;
	};

struct PhaseScanArgs
	{
	const PhaseSeg * seg;       // [C][segs_per_channel][B]
	int segs_per_channel, B;
	int group_len, groups;      // segments per scan group, ceil(segs_per_channel / group_len) <= 65535
	PhaseSeg * group;           // [C][groups][B] scratch
	const PhaseSeg * carry_in;  // [C][B] or null (state before the first local frame)
	PhaseSeg * carry_out;       // [C][B] or null (state after the last local frame)
	double * acc_start;         // [C][segs_per_channel][B] or null
	double P, rcpP;
	// expand_only: `group` already holds the exclusive prefixes of a scan that ran WITHOUT a carry (a summary-only call on
	// the same data); only the re-walk runs, entering every group through expand_carry (+) prefix (the combine is exact
	// and associative, DESIGN.md 4.2, so the result has the bits of the scan with carry_in == expand_carry)
	int expand_only;
	const PhaseSeg * expand_carry;   // [C][B] or null
	// fix_pv != null: summaries left by the analysis kernel (analysis_cta<EMIT>); entries it could not produce carry a NaN
	// marker and are recomputed here, in the group reduction, from the rows -- and written back for the re-walk
	const float2 * fix_pv; int64_t fix_channel_stride, fix_frame_begin, fix_frame_end; int fix_seg_len;
	PvConsts fix_k; int * fix_nan_flag;
	};

// The transform kernels this build carries (pv_kernel_list.h), by the descriptor the launch policy (pv_policy.h)
// returns. A descriptor the build does not carry, or one of the other stage, gives cudaErrorInvalidValue.
cudaError_t launch( const TransformKernel & k, const AnalysisArgs & a, int64_t blocks, cudaStream_t st );
cudaError_t launch( const TransformKernel & k, const SynthArgs & a, int64_t blocks, cudaStream_t st );
// The kernel's resident CTAs per SM with these arguments' shared memory (the pipelined host forms cut a signal into
// slices of whole waves). Kernels that allocate tensor memory: what their registers and columns admit.
cudaError_t resident_ctas( const TransformKernel & k, const AnalysisArgs & a, int * ctas );
cudaError_t resident_ctas( const TransformKernel & k, const SynthArgs & a, int * ctas );
cudaError_t launch_phase_seg( const PhaseSegArgs & a, int C, cudaStream_t st );
cudaError_t launch_phase_scan( const PhaseScanArgs & a, int C, cudaStream_t st );
cudaError_t launch_phase_carry( const PhaseSeg * all, int rank, int64_t per_rank, PhaseSeg * carry, double P, double rcpP, cudaStream_t st );
cudaError_t launch_mid_side( const float * in, float * out, int64_t n, int sms, cudaStream_t st );
cudaError_t launch_zero_shared( float * out, int64_t out_stride, int64_t out_offset, int64_t out_len, int C,
                                int64_t frame_begin, int64_t frame_end, int seg_len, int segs, int W, int hop, cudaStream_t st );
cudaError_t launch_add( float * out, const float * add, int64_t n, int sms, cudaStream_t st );


// One launch pushes a phase state to several peers: CTA b copies `n16` 16-byte units from src to dst[b] (peer memory over
// NVLink: P2P access enabled or an IPC mapping) and then, when count[b] is set, increments that peer's arrival counter at
// system scope. Fourteen DMA operations in a row -- a copy and a flag per destination -- took ~14 us per destination.
struct StatePush
	{
	const uint4 * src; unsigned n16;
	uint4 * dst[16]; unsigned * count[16];
	};
cudaError_t launch_state_push( const StatePush & p, int destinations, cudaStream_t st );

} // namespace pvk
