// flan_b200/csrc/pv_modify.cu -- sm_100a kernels of the PV-domain chain between analysis and resynthesis:
// PV::repitch / PV::modify_frequency (reference PV/PVModify.cpp:196-305) and PV::stretch / PV::modify_time
// (PVModify.cpp:307-385). Bodies in pv_modify_body.cuh. Compiled with -fmad=false: results are bit-identical to the
// reference's float arithmetic. All of them stream MF rows once: HBM-bound integer / float work, no tensor cores.
#include "pv_modify.h"

namespace pvm {

// One CTA per (channel, frame) row: stage the row in shared memory, map, scatter, store. Algorithmic bytes per row:
// 8B read + 8B written (+ 4B of table when it is not shared between frames, + 4B for modify_frequency's in_mod).
__global__ void __launch_bounds__( 256 ) pv_repitch_kernel( const RepitchArgs a, int64_t rows, const int * skip_if )
	{
	extern __shared__ __align__( 16 ) unsigned char smem[];
	if( skip_if && *skip_if ) return;
	RepitchRow s( smem, a.B );
	const int tid = threadIdx.x, nt = blockDim.x;
	for( int64_t row = blockIdx.x; row < rows; row += gridDim.x )
		{
		repitch_load( a, row, tid, nt, s );
		__syncthreads();
		const int mine = repitch_map( a, tid, nt, s );
		const int down = __syncthreads_or( mine & 1 );
		const int up = __syncthreads_or( mine & 2 );
		repitch_scatter( a, ( down ? 1 : 0 ) | ( up ? 2 : 0 ), tid, nt, s );
		__syncthreads();
		repitch_store( a, row, tid, nt, s );
		__syncthreads();
		}
	}

// Running sums along bins are sequential per row (float addition does not re-associate): one lane per row, rows
// staged through shared memory in 32 x 32 tiles so that global loads and stores stay coalesced.
__global__ void __launch_bounds__( 256 ) pv_bin_prefix_kernel( const Table factor, int64_t rows, int B, float sample_rate, float dft, float * out )
	{
	__shared__ float tile[8][32][33];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const int64_t row0 = ( (int64_t) blockIdx.x * 8 + warp ) * 32;
	if( row0 >= rows ) return;
	float acc = 0.0f;
	for( int b0 = 0; b0 < B; b0 += 32 )
		{
		for( int r = 0; r < 32; ++r )
			if( row0 + r < rows && b0 + lane < B ) tile[warp][r][lane] = factor.at( row0 + r, b0 + lane );
		__syncwarp();
		if( row0 + lane < rows )
			for( int j = 0; j < 32 && b0 + j < B; ++j )
				{
				const float v = tile[warp][lane][j];
				acc = ( b0 + j == 0 ) ? v : v + acc;
				tile[warp][lane][j] = acc * sample_rate / dft;          // PVBuffer.cpp:443-446
				}
		__syncwarp();
		for( int r = 0; r < 32; ++r )
			if( row0 + r < rows && b0 + lane < B ) out[( row0 + r ) * B + b0 + lane] = tile[warp][r][lane];
		__syncwarp();
		}
	}

__global__ void pv_frame_prefix_kernel( const Table factor, int64_t F, int cols, float * raw )
	{
	const int col = blockIdx.x * blockDim.x + threadIdx.x;
	if( col >= cols ) return;
	frame_prefix_column( factor, col, F, cols, raw );
	}

__global__ void pv_frame_convert_kernel( const float * raw, float * out, int64_t total, float rate )
	{
	for( int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t) gridDim.x * blockDim.x )
		frame_prefix_convert( raw, out, i, rate );
	}

__global__ void pv_map_check_kernel( const Table mod, int64_t F, int cols, MapCheck * check )
	{
	const int64_t total = F * cols;
	float mx = 0.0f; bool any = false, down = false;
	for( int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t) gridDim.x * blockDim.x )
		{
		float sec; bool d;
		time_map_check( mod, i / cols, (int)( i % cols ), sec, d );
		if( !any || mx < sec ) mx = sec;
		any = true; down |= d;
		}
	unsigned int key = any ? float_key( mx ) : 0u;
	for( int o = 16; o; o >>= 1 ) { const unsigned int k = __shfl_xor_sync( 0xffffffffu, key, o ); key = k > key ? k : key; }
	down = __any_sync( 0xffffffffu, down );
	if( ( threadIdx.x & 31 ) == 0 )
		{
		if( key ) atomicMax( &check->max_key, key );
		if( down ) check->descends = 1;
		}
	}

// thread = (channel, chunk of frame pairs, bin): reads 8 bytes per input MF once (plus one overlap frame per chunk),
// writes every output MF once. Adjacent lanes = adjacent bins: row segments are coalesced on both sides whenever the
// time map is shared between bins.
__global__ void __launch_bounds__( 128 ) pv_stretch_kernel( const StretchArgs a, int bin_tiles )
	{
	const int64_t blk = blockIdx.x;
	const int bin = (int)( blk % bin_tiles ) * 128 + threadIdx.x;
	const int64_t chunk_index = blk / bin_tiles;
	if( bin >= a.B ) return;
	stretch_chunk( a, blockIdx.y, chunk_index, bin );
	}

__global__ void __launch_bounds__( 128 ) pv_stretch_seq_kernel( const StretchArgs a )
	{
	const int bin = blockIdx.x * 128 + threadIdx.x;
	if( bin >= a.B ) return;
	stretch_column( a, blockIdx.y, bin );
	}

// ---- constant factor: closed-form running sum (see constant_prefix_segments) ---------------------------------------
__global__ void pv_constant_prefix_kernel( const float * factor, int64_t F, PrefixSeg * segs, int * count )
	{
	*count = constant_prefix_segments( *factor, F, segs );
	}

__global__ void pv_constant_fill_kernel( const float * factor, int64_t F, const PrefixSeg * segs, const int * count, float rate, float * out )
	{
	__shared__ PrefixSeg s_segs[PREFIX_MAX_SEGS];
	const int ns = *count < PREFIX_MAX_SEGS ? *count : PREFIX_MAX_SEGS;
	for( int i = threadIdx.x; i < ns; i += blockDim.x ) s_segs[i] = segs[i];
	__syncthreads();
	const float c = *factor;
	for( int64_t k = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; k < F; k += (int64_t) gridDim.x * blockDim.x )
		out[k] = constant_prefix_value( s_segs, ns, c, k ) / rate;      // frame_to_time, PVBuffer.cpp:433-436
	}

// ---- frame-shared repitch: plan + gather ------------------------------------------------------------------------
__global__ void __launch_bounds__( 1024 ) pv_repitch_plan_kernel( const float * hz, int B, float bin_width, int interp, const RepitchPlan plan )
	{
	extern __shared__ __align__( 16 ) unsigned char smem[];
	float * pos = (float *) smem;
	const int tid = threadIdx.x, nt = blockDim.x;
	repitch_plan_positions( hz, B, bin_width, tid, nt, pos, plan );
	__syncthreads();
	const int mine = repitch_plan_flags( B, tid, nt, pos );
	const int down = __syncthreads_or( mine & 1 );
	const int up = __syncthreads_or( mine & 2 );
	repitch_plan_pairs( B, interp, ( down ? 1 : 0 ) | ( up ? 2 : 0 ), tid, nt, pos, plan );
	}

// Persistent CTAs, one row at a time: the row's (m, f) pairs are loaded one row ahead into registers, the mapped
// frequencies go through a double-buffered shared-memory row (one barrier per row), every output bin is one gather.
// Algorithmic bytes per row: 8B read + 8B written; the plan (12B bytes) lives in shared memory for the CTA's lifetime.
constexpr int REPITCH_J = 5;        // bins per thread
template<int T> __global__ void __launch_bounds__( T ) pv_repitch_shared_kernel( const RepitchArgs a, const RepitchPlan plan, const float * hz, int64_t rows )
	{
	extern __shared__ __align__( 16 ) unsigned char smem[];
	if( !*plan.ok ) return;
	const int B = a.B, tid = threadIdx.x;
	int * src = (int *) smem;
	float * mix = (float *)( src + B );
	float * hzs = mix + B;
	float * mbuf = hzs + B;          // [2][B]
	float * fbuf = mbuf + 2 * B;     // [2][B]
	for( int b = tid; b < B; b += T ) { src[b] = plan.src[b]; mix[b] = plan.mix[b]; hzs[b] = hz[b]; }
	__syncthreads();
	float2 reg[REPITCH_J];
	int64_t row = blockIdx.x;
	if( row < rows )
		{
#pragma unroll
		for( int j = 0; j < REPITCH_J; ++j ) { const int b = tid + j * T; if( b < B ) reg[j] = __ldcs( a.pv + row * B + b ); }
		}
	for( int k = 0; row < rows; row += gridDim.x, k ^= 1 )
		{
		float * m = mbuf + k * B, * fm = fbuf + k * B;
#pragma unroll
		for( int j = 0; j < REPITCH_J; ++j )
			{
			const int b = tid + j * T;
			if( b < B )
				{
				m[b] = reg[j].x;
				fm[b] = a.in_mod ? __ldcs( a.in_mod + row * B + b ) : repitch_lerp( hzs, B, a.bin_width, reg[j].y );
				}
			}
		const int64_t next = row + gridDim.x;
		if( next < rows )
			{
#pragma unroll
			for( int j = 0; j < REPITCH_J; ++j ) { const int b = tid + j * T; if( b < B ) reg[j] = __ldcs( a.pv + next * B + b ); }
			}
		__syncthreads();
		float2 * out = a.out + row * B;
#pragma unroll
		for( int j = 0; j < REPITCH_J; ++j )
			{
			const int y = tid + j * T;
			if( y < B ) __stcs( out + y, repitch_gather( y, src, mix, m, fm ) );
			}
		}
	}

// ---- bin-shared stretch: plan + chunk walk ----------------------------------------------------------------------
__global__ void pv_stretch_plan_kernel( const StretchArgs a, const StretchPlan plan )
	{
	const int64_t f = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	if( f < a.F ) stretch_plan_frame( a, plan, f );
	}

// thread = (channel, segment of seg_len OUTPUT frames, bin); summ.seg_out != null: also the segment's phase summary, laid
// out like pv_phase_seg_kernel's ([C][segs][B]), and the NaN / Inf flag of AudioPV.cpp:88
template<bool SUMM>
__global__ void __launch_bounds__( 128 ) pv_stretch_planned_kernel( const StretchArgs a, const StretchPlan plan, const StretchSummary summ, int bin_tiles )
	{
	const int64_t blk = blockIdx.x;
	const int bin = (int)( blk % bin_tiles ) * 128 + threadIdx.x;
	const int64_t seg = blk / bin_tiles;
	if( bin >= a.B ) return;
	pvk::PhaseSegAcc acc;
	stretch_segment_planned<SUMM>( a, plan, blockIdx.y, seg, summ.seg_len, bin, &acc, summ.k );
	if( SUMM )
		{
		summ.seg_out[( (int64_t) blockIdx.y * summ.segs_per_channel + seg ) * a.B + bin] = acc.finish( summ.P, summ.rcpP );
		if( acc.bad ) *summ.nan_flag = 1;
		}
	}

bool repitch_shared_supported( int B ) { return B <= REPITCH_J * 1024; }

cudaError_t launch_repitch_plan( const float * hz, int B, float bin_width, int interp, const RepitchPlan & plan, cudaStream_t st )
	{
	pv_repitch_plan_kernel<<<1, 1024, sizeof( float ) * B, st>>>( hz, B, bin_width, interp, plan );
	return cudaGetLastError();
	}

template<int T> static cudaError_t launch_repitch_shared_t( const RepitchArgs & a, const RepitchPlan & plan, const float * hz, int64_t rows, int sms, cudaStream_t st )
	{
	const size_t smem = sizeof( float ) * 7 * (size_t) a.B;
	cudaError_t e = cudaFuncSetAttribute( pv_repitch_shared_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem );
	if( e != cudaSuccess ) return e;
	int per_sm = 0;
	e = cudaOccupancyMaxActiveBlocksPerMultiprocessor( &per_sm, pv_repitch_shared_kernel<T>, T, smem );
	if( e != cudaSuccess ) return e;
	if( per_sm < 1 ) per_sm = 1;
	int64_t blocks = (int64_t) sms * per_sm;
	if( blocks > rows ) blocks = rows;
	pv_repitch_shared_kernel<T><<<(unsigned) blocks, T, smem, st>>>( a, plan, hz, rows );
	return cudaGetLastError();
	}

cudaError_t launch_repitch_shared( const RepitchArgs & a, const RepitchPlan & plan, const float * hz, int64_t rows, int sms, cudaStream_t st )
	{
	if( a.B <= REPITCH_J * 256 ) return launch_repitch_shared_t<256>( a, plan, hz, rows, sms, st );
	if( a.B <= REPITCH_J * 512 ) return launch_repitch_shared_t<512>( a, plan, hz, rows, sms, st );
	return launch_repitch_shared_t<1024>( a, plan, hz, rows, sms, st );
	}

__global__ void pv_stretch_window_kernel( const StretchPlan plan, int64_t F, const StretchWindows w, int64_t * rows )
	{
	const int i = threadIdx.x;
	if( i < w.n ) stretch_window( plan, F, w.xb[i], w.xb[i + 1], rows + 2 * i, rows + 2 * i + 1 );
	}

cudaError_t launch_stretch_plan( const StretchArgs & a, const StretchPlan & plan, cudaStream_t st )
	{
	cudaError_t e = cudaMemsetAsync( plan.src, 0xff, sizeof( int ) * (size_t) a.out_frames, st );      // -1: no pair covers the frame
	if( e != cudaSuccess ) return e;
	pv_stretch_plan_kernel<<<(unsigned)( ( a.F + 127 ) / 128 ), 128, 0, st>>>( a, plan );
	return cudaGetLastError();
	}

cudaError_t launch_stretch_windows( const StretchPlan & plan, int64_t F, const StretchWindows & w, int64_t * rows, cudaStream_t st )
	{
	if( w.n < 1 || w.n > StretchWindows::MAX ) return cudaErrorInvalidValue;
	pv_stretch_window_kernel<<<1, 32, 0, st>>>( plan, F, w, rows );
	return cudaGetLastError();
	}

cudaError_t launch_stretch_segments( const StretchArgs & a, const StretchPlan & plan, const StretchSummary & summ, int C, cudaStream_t st )
	{
	const int bin_tiles = ( a.B + 127 ) / 128;
	const int64_t blocks = (int64_t) summ.segs_per_channel * bin_tiles;
	if( blocks > 0x7fffffff || summ.seg_len < 1 ) return cudaErrorInvalidValue;
	if( blocks == 0 ) return cudaSuccess;
	if( summ.seg_out ) pv_stretch_planned_kernel<true><<<dim3( (unsigned) blocks, C ), 128, 0, st>>>( a, plan, summ, bin_tiles );
	else pv_stretch_planned_kernel<false><<<dim3( (unsigned) blocks, C ), 128, 0, st>>>( a, plan, summ, bin_tiles );
	return cudaGetLastError();
	}

cudaError_t launch_stretch_planned( const StretchArgs & a, const StretchPlan & plan, const StretchSummary & summ, int C, cudaStream_t st )
	{
	const int bin_tiles = ( a.B + 127 ) / 128;
	if( (int64_t) summ.segs_per_channel * bin_tiles > 0x7fffffff || summ.seg_len < 1 ) return cudaErrorInvalidValue;
	const cudaError_t e = launch_stretch_plan( a, plan, st );
	if( e != cudaSuccess ) return e;
	return launch_stretch_segments( a, plan, summ, C, st );
	}

cudaError_t launch_bin_prefix( const Table & factor, int64_t rows, int B, float sample_rate, float dft, float * out, cudaStream_t st )
	{
	const int64_t blocks = ( rows + 255 ) / 256;
	pv_bin_prefix_kernel<<<(unsigned) blocks, 256, 0, st>>>( factor, rows, B, sample_rate, dft, out );
	return cudaGetLastError();
	}

cudaError_t launch_frame_prefix( const Table & factor, int64_t F, int cols, float rate, float * raw_scratch, float * out, int sms, cudaStream_t st )
	{
	pv_frame_prefix_kernel<<<( cols + 63 ) / 64, 64, 0, st>>>( factor, F, cols, raw_scratch );
	int64_t blocks = ( F * cols + 255 ) / 256;
	if( blocks > (int64_t) sms * 8 ) blocks = (int64_t) sms * 8;
	pv_frame_convert_kernel<<<(unsigned) blocks, 256, 0, st>>>( raw_scratch, out, F * cols, rate );
	return cudaGetLastError();
	}

cudaError_t launch_constant_prefix( const float * factor, int64_t F, float rate, void * scratch, float * out, int sms, cudaStream_t st )
	{
	PrefixSeg * segs = (PrefixSeg *) scratch;
	int * count = (int *)( segs + PREFIX_MAX_SEGS );
	pv_constant_prefix_kernel<<<1, 1, 0, st>>>( factor, F, segs, count );
	int64_t blocks = ( F + 255 ) / 256;
	if( blocks > (int64_t) sms * 4 ) blocks = (int64_t) sms * 4;
	pv_constant_fill_kernel<<<(unsigned) blocks, 256, 0, st>>>( factor, F, segs, count, rate, out );
	return cudaGetLastError();
	}

cudaError_t launch_map_check( const Table & mod, int64_t F, int cols, MapCheck * check, int sms, cudaStream_t st )
	{
	cudaError_t e = cudaMemsetAsync( check, 0, sizeof( MapCheck ), st );
	if( e != cudaSuccess ) return e;
	int64_t blocks = ( F * cols + 255 ) / 256;
	if( blocks > (int64_t) sms * 8 ) blocks = (int64_t) sms * 8;
	if( blocks < 1 ) blocks = 1;
	pv_map_check_kernel<<<(unsigned) blocks, 256, 0, st>>>( mod, F, cols, check );
	return cudaGetLastError();
	}

cudaError_t launch_repitch( const RepitchArgs & a, int64_t rows, const int * skip_if, cudaStream_t st )
	{
	const size_t smem = RepitchRow::bytes( a.B );
	cudaError_t e = cudaFuncSetAttribute( pv_repitch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem );
	if( e != cudaSuccess ) return e;
	const int64_t blocks = rows < 0x7fffffff ? rows : 0x7fffffff;
	pv_repitch_kernel<<<(unsigned) blocks, 256, smem, st>>>( a, rows, skip_if );
	return cudaGetLastError();
	}

cudaError_t launch_stretch_parallel( const StretchArgs & a, int C, cudaStream_t st )
	{
	const int bin_tiles = ( a.B + 127 ) / 128;
	const int64_t blocks = a.chunks * bin_tiles;
	if( blocks > 0x7fffffff ) return cudaErrorInvalidValue;
	pv_stretch_kernel<<<dim3( (unsigned) blocks, C ), 128, 0, st>>>( a, bin_tiles );
	return cudaGetLastError();
	}

cudaError_t launch_stretch_sequential( const StretchArgs & a, int C, cudaStream_t st )
	{
	pv_stretch_seq_kernel<<<dim3( ( a.B + 127 ) / 128, C ), 128, 0, st>>>( a );
	return cudaGetLastError();
	}

} // namespace pvm
