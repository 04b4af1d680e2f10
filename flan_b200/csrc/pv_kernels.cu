// flan_b200/csrc/pv_kernels.cu -- sm_100a kernels of the phase-vocoder engine and their launchers.
//
//   pv_analysis_kernel<N>    Audio::convert_to_PV     (reference Conversions/AudioPV.cpp:12-78)
//   pv_phase_seg_kernel      per-segment phase-sum summaries     (phase_vocoder.cpp:57-59, scan form)
//   pv_phase_scan_kernel     exclusive scan of the summaries over segments -> accumulator per segment
//   pv_synthesis_kernel<N>   PV::convert_to_audio     (AudioPV.cpp:86-139)
//   pv_mid_side_kernel       Audio::convert_to_mid_side (Audio/AudioConversions.cpp:32-51)
//
// The CTA bodies live in pv_body.cuh (shared with the CPU thread emulator); this file supplies the
// device Env (barrier, cp.async staging, cache-hinted loads/stores, red.add) and the launch geometry.
#include "pv_body.cuh"
#include "pv_launch.h"
#include "pv_kernel_list.h"

#include <cuda_runtime.h>

#include <cstdlib>
#include <type_traits>
#include <vector>

namespace pvk {

struct DeviceEnv
	{
	int tid;
	__device__ __forceinline__ void syncwarp() { __syncwarp(); }
	__device__ __forceinline__ bool any( bool p ) { return __any_sync( 0xffffffffu, p ); }
	__device__ __forceinline__ void sync()
		{
#ifndef PV_ABL_NOSYNC
		__syncthreads();
#endif
		}
	__device__ __forceinline__ float ldg( const float * p ) { return __ldg( p ); }
	__device__ __forceinline__ float2 ldg2( const float2 * p ) { return __ldg( p ); }
	__device__ __forceinline__ float4 ldg4( const float4 * p ) { return __ldg( p ); }
	__device__ __forceinline__ float2 ldcs2( const float2 * p ) { return __ldcs( p ); }
	// streaming stores that do not allocate in L1 (STG.E.NA): the PV rows and output samples would otherwise push the
	// window samples and the tables out of it (measured against st.global.cs: analysis 1.685 -> 1.660 ms on cfg2)
	__device__ __forceinline__ void st_stream2( float2 * p, float2 v )
		{ asm volatile( "st.global.L1::no_allocate.v2.f32 [%0], {%1, %2};" :: "l"( p ), "f"( v.x ), "f"( v.y ) : "memory" ); }
	__device__ __forceinline__ void st_stream( float * p, float v ) { __stcs( p, v ); }
	__device__ __forceinline__ void red_add( float * p, float v ) { atomicAdd( p, v ); }
	// shared-memory word += v without a round trip through registers (the word is private to the calling thread)
	__device__ __forceinline__ void shared_add( int * p, int v ) { asm volatile( "red.shared.add.s32 [%0], %1;" :: "r"( (unsigned) __cvta_generic_to_shared( p ) ), "r"( v ) : "memory" ); }
	// 8-byte asynchronous global->shared copy (LDGSTS), completion tracked per thread by commit / wait groups
	__device__ __forceinline__ void cp_async8( float2 * dst, const float2 * src )
		{
		const unsigned d = (unsigned) __cvta_generic_to_shared( dst );
		asm volatile( "cp.async.ca.shared.global [%0], [%1], 8;\n" :: "r"( d ), "l"( src ) : "memory" );
		}
	__device__ __forceinline__ void cp_async_commit() { asm volatile( "cp.async.commit_group;\n" ::: "memory" ); }
	__device__ __forceinline__ void cp_async_wait_all() { asm volatile( "cp.async.wait_group 0;\n" ::: "memory" ); }
	// Bulk (TMA) global->shared copy tracked by an mbarrier: one thread arms the barrier with the byte count and issues
	// the copy; every thread waits on the phase parity. Addresses and size are multiples of 16 bytes.
	typedef unsigned long long BulkBarrier;
	__device__ __forceinline__ void bulk_init( BulkBarrier * bar )
		{
		const unsigned b = (unsigned) __cvta_generic_to_shared( bar );
		asm volatile( "mbarrier.init.shared::cta.b64 [%0], 1;\n" :: "r"( b ) : "memory" );
		asm volatile( "fence.mbarrier_init.release.cluster;\n" ::: "memory" );
		}
	__device__ __forceinline__ void bulk_load( void * dst, const void * src, unsigned bytes, BulkBarrier * bar )
		{
		const unsigned b = (unsigned) __cvta_generic_to_shared( bar );
		const unsigned d = (unsigned) __cvta_generic_to_shared( dst );
		asm volatile( "mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" :: "r"( b ), "r"( bytes ) : "memory" );
		asm volatile( "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
		              :: "r"( d ), "l"( src ), "r"( bytes ), "r"( b ) : "memory" );
		}
	__device__ __forceinline__ void bulk_wait( BulkBarrier * bar, unsigned parity )
		{
		const unsigned b = (unsigned) __cvta_generic_to_shared( bar );
		asm volatile(
			"{\n"
			".reg .pred p;\n"
			"WAIT_%=:\n"
			"mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
			"@p bra DONE_%=;\n"
			"bra WAIT_%=;\n"
			"DONE_%=:\n"
			"}\n" :: "r"( b ), "r"( parity ) : "memory" );
		}
#ifdef PV_PREFETCH_L1
	__device__ __forceinline__ void prefetch( const void * p ) { asm volatile( "prefetch.global.L1 [%0];" :: "l"( p ) ); }
#else
	__device__ __forceinline__ void prefetch( const void * p ) { asm volatile( "prefetch.global.L2 [%0];" :: "l"( p ) ); }
#endif
	// Tensor memory as per-thread storage (no MMA): `tmem` is the CTA's allocation plus this warp's lane quarter, so
	// column j of the calling thread is word j of its private row. tcgen05.ld / .st are .sync.aligned: every lane of the
	// warp issues them together. A load's registers are defined only after tmem_wait, which also ties them to it so
	// that no use can be scheduled above the wait. A column this thread stored is read back only after a tmem_wait_st
	// that follows the store (tcgen05.st and tcgen05.ld of one thread are not ordered with each other otherwise); the
	// emulator (emu/pv_emu.cpp) aborts on a load that breaks this. Stores and waits carry no memory clobber either.
	uint32_t tmem;
	template<int K> __device__ __forceinline__ void tmem_st( int col, const float * r )
		{
		const uint32_t a = tmem + (uint32_t) col;
		if constexpr( K == 2 )
			asm volatile( "tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1,%2};" :: "r"( a ), "f"( r[0] ), "f"( r[1] ) );
		else if constexpr( K == 4 )
			asm volatile( "tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" :: "r"( a ), "f"( r[0] ), "f"( r[1] ), "f"( r[2] ), "f"( r[3] ) );
		else if constexpr( K == 8 )
			asm volatile( "tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
			              :: "r"( a ), "f"( r[0] ), "f"( r[1] ), "f"( r[2] ), "f"( r[3] ), "f"( r[4] ), "f"( r[5] ), "f"( r[6] ), "f"( r[7] ) );
		else if constexpr( K == 16 )
			asm volatile( "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
			              :: "r"( a ), "f"( r[0] ), "f"( r[1] ), "f"( r[2] ), "f"( r[3] ), "f"( r[4] ), "f"( r[5] ), "f"( r[6] ), "f"( r[7] ),
			                 "f"( r[8] ), "f"( r[9] ), "f"( r[10] ), "f"( r[11] ), "f"( r[12] ), "f"( r[13] ), "f"( r[14] ), "f"( r[15] ) );
		else if constexpr( K == 32 )
			asm volatile( "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,"
			              "%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
			              :: "r"( a ),
			                 "f"( r[0] ), "f"( r[1] ), "f"( r[2] ), "f"( r[3] ), "f"( r[4] ), "f"( r[5] ), "f"( r[6] ), "f"( r[7] ),
			                 "f"( r[8] ), "f"( r[9] ), "f"( r[10] ), "f"( r[11] ), "f"( r[12] ), "f"( r[13] ), "f"( r[14] ), "f"( r[15] ),
			                 "f"( r[16] ), "f"( r[17] ), "f"( r[18] ), "f"( r[19] ), "f"( r[20] ), "f"( r[21] ), "f"( r[22] ), "f"( r[23] ),
			                 "f"( r[24] ), "f"( r[25] ), "f"( r[26] ), "f"( r[27] ), "f"( r[28] ), "f"( r[29] ), "f"( r[30] ), "f"( r[31] ) );
		else static_assert( K == 2, "tcgen05.st widths 2, 4, 8, 16, 32" );
		}
	__device__ __forceinline__ void tmem_wait_st() { asm volatile( "tcgen05.wait::st.sync.aligned;" ); }
	template<int K> __device__ __forceinline__ void tmem_ld( int col, float * r )
		{
		const uint32_t a = tmem + (uint32_t) col;
		if constexpr( K == 2 )
			asm volatile( "tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0,%1}, [%2];" : "=f"( r[0] ), "=f"( r[1] ) : "r"( a ) );
		else if constexpr( K == 4 )
			asm volatile( "tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];" : "=f"( r[0] ), "=f"( r[1] ), "=f"( r[2] ), "=f"( r[3] ) : "r"( a ) );
		else if constexpr( K == 8 )
			asm volatile( "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
			              : "=f"( r[0] ), "=f"( r[1] ), "=f"( r[2] ), "=f"( r[3] ), "=f"( r[4] ), "=f"( r[5] ), "=f"( r[6] ), "=f"( r[7] ) : "r"( a ) );
		else if constexpr( K == 16 )
			asm volatile( "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
			              : "=f"( r[0] ), "=f"( r[1] ), "=f"( r[2] ), "=f"( r[3] ), "=f"( r[4] ), "=f"( r[5] ), "=f"( r[6] ), "=f"( r[7] ),
			                "=f"( r[8] ), "=f"( r[9] ), "=f"( r[10] ), "=f"( r[11] ), "=f"( r[12] ), "=f"( r[13] ), "=f"( r[14] ), "=f"( r[15] ) : "r"( a ) );
		else if constexpr( K == 32 )
			asm volatile( "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,"
			              "%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
			              : "=f"( r[0] ), "=f"( r[1] ), "=f"( r[2] ), "=f"( r[3] ), "=f"( r[4] ), "=f"( r[5] ), "=f"( r[6] ), "=f"( r[7] ),
			                "=f"( r[8] ), "=f"( r[9] ), "=f"( r[10] ), "=f"( r[11] ), "=f"( r[12] ), "=f"( r[13] ), "=f"( r[14] ), "=f"( r[15] ),
			                "=f"( r[16] ), "=f"( r[17] ), "=f"( r[18] ), "=f"( r[19] ), "=f"( r[20] ), "=f"( r[21] ), "=f"( r[22] ), "=f"( r[23] ),
			                "=f"( r[24] ), "=f"( r[25] ), "=f"( r[26] ), "=f"( r[27] ), "=f"( r[28] ), "=f"( r[29] ), "=f"( r[30] ), "=f"( r[31] ) : "r"( a ) );
		else static_assert( K == 2, "tcgen05.ld widths 2, 4, 8, 16, 32" );
		}
	// waits for every outstanding tmem_ld of the thread; the K registers at r are the ones its callers go on to use.
	// The loads and the wait carry no memory clobber: they touch no memory the compiler sees, so shared- and global-memory
	// accesses may be scheduled across them.
	template<int K> __device__ __forceinline__ void tmem_wait( float * r )
		{
		asm volatile( "tcgen05.wait::ld.sync.aligned;" );
#pragma unroll
		for( int i = 0; i < K; ++i ) asm volatile( "" : "+f"( r[i] ) );
		}
	};

// Tensor-memory lifetime of one CTA (128-thread bodies, COLS columns per thread). Warp 0 allocates and gives up its
// permit to allocate again, the fences order the allocation's shared-memory result around the barrier, and a final
// barrier on every path precedes the deallocation: a CTA that exited holding columns would leave the SM unable to
// allocate them. The bodies return to the kernel wrapper on every path (the early return of an empty segment too).
template<int COLS> struct TmemScope
	{
	static_assert( COLS >= 32 && COLS <= 512 && ( COLS & ( COLS - 1 ) ) == 0, "tcgen05.alloc takes a power of two >= 32 columns" );
	uint32_t * slot;
	__device__ __forceinline__ explicit TmemScope( uint32_t * s ) : slot( s )
		{
		if( threadIdx.x < 32 )
			{
			asm volatile( "tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"( (unsigned) __cvta_generic_to_shared( slot ) ), "n"( COLS ) : "memory" );
			asm volatile( "tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory" );
			}
		asm volatile( "tcgen05.fence::before_thread_sync;" ::: "memory" );
		__syncthreads();
		asm volatile( "tcgen05.fence::after_thread_sync;" ::: "memory" );
		}
	__device__ __forceinline__ uint32_t base() const { return *slot + ( ( threadIdx.x & 96u ) << 16 ); }   // this warp's 32 lanes
	__device__ __forceinline__ ~TmemScope()
		{
		asm volatile( "tcgen05.fence::before_thread_sync;" ::: "memory" );
		__syncthreads();
		asm volatile( "tcgen05.fence::after_thread_sync;" ::: "memory" );
		if( threadIdx.x < 32 ) asm volatile( "tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"( *slot ), "n"( COLS ) : "memory" );
		}
	};

// TPS = resident threads per SM the register allocation is sized for (512 -> 128, 768 -> 85, 1024 -> 64 registers).
constexpr int min_blocks( int threads, int TPS ) { return TPS / threads > 32 ? 32 : ( TPS / threads > 0 ? TPS / threads : 1 ); }

// The analysis instantiations that keep their loop invariants in tensor memory: those whose register budget admits no
// more CTAs per SM than 512 columns serve (development builds also carry 5- and 6-CTA variants, which keep the L1 form).
template<int N, int PT, int TPS> constexpr bool analysis_uses_tmem()
	{
	return analysis_tmem<N, PT>() && min_blocks( N / ( 2 * PT ), TPS ) * AN_TM_COLS <= 512;
	}

template<int N, int TPS, bool GEN> constexpr bool synthesis_uses_tmem()
	{
	return synthesis_tmem<N, GEN>() && min_blocks( N / 32, TPS ) * SY_TM_COLS <= 512;
	}

// PT = complex points per thread: 8 (radix-8 passes, N/16 threads per frame) or 16 (radix-16 passes, N/32 threads).
template<int N, int PT, int TPS, bool ONE, bool PAD = false, bool EMIT = false>
__global__ void __launch_bounds__( N / ( 2 * PT ), min_blocks( N / ( 2 * PT ), TPS ) ) pv_analysis_kernel( const AnalysisArgs a )
	{
	extern __shared__ __align__( 16 ) unsigned char smem_raw[];
	float2 * x0 = reinterpret_cast<float2 *>( smem_raw );
	float2 * x1 = ONE ? x0 : x0 + XBuf<N / 2>::size;
	constexpr bool TM = analysis_uses_tmem<N, PT, TPS>();
	// N/2 + 1 per-bin sums (EMIT only; TM: in tensor memory)
	int * ssum = EMIT && !TM ? reinterpret_cast<int *>( x1 + XBuf<N / 2>::size ) : nullptr;
	DeviceEnv env; env.tid = threadIdx.x;
	if constexpr( TM )
		{
		__shared__ uint32_t tmem_slot;
		TmemScope<AN_TM_COLS> scope( &tmem_slot );
		env.tmem = scope.base();
		analysis_cta<N, PT, ONE, PAD, EMIT, true>( a, (int64_t) blockIdx.x, env, x0, x1, ssum );
		}
	else analysis_cta<N, PT, ONE, PAD, EMIT, false>( a, (int64_t) blockIdx.x, env, x0, x1, ssum );
	}

// Mirrored last pass (pv_body.cuh: analysis_cta_mirror): 16 points per thread, unpack + phase vocoder on the thread's own registers.
template<int N, int TPS>
__global__ void __launch_bounds__( N / 32, min_blocks( N / 32, TPS ) ) pv_analysis_mirror_kernel( const AnalysisArgs a )
	{
	extern __shared__ __align__( 16 ) unsigned char smem_raw[];
	float2 * x0 = reinterpret_cast<float2 *>( smem_raw );
	float2 * x1 = a.one_buffer ? x0 : x0 + XBuf<N / 2>::size;
	float2 * ring = x1 + XBuf<N / 2>::size;            // N/2 pairs: the window's samples, thread-private entries
	float2 * scratch = ring + N / 2;                   // 16 pairs
	DeviceEnv env; env.tid = threadIdx.x;
	analysis_cta_mirror<N>( a, (int64_t) blockIdx.x, env, x0, x1, ring, scratch );
	}

template<int N, int TPS, bool ONE>
__global__ void __launch_bounds__( N / 16, min_blocks( N / 16, TPS ) ) pv_synthesis_kernel( const SynthArgs a )
	{
	extern __shared__ __align__( 16 ) unsigned char smem_raw[];
	float * ola = reinterpret_cast<float *>( smem_raw );
	float2 * x0 = reinterpret_cast<float2 *>( smem_raw + sizeof( float ) * N );
	float2 * x1 = ONE ? x0 : x0 + XBuf<N / 2>::size;
	float2 * rowbuf = x1 + XBuf<N / 2>::size;
	DeviceEnv env; env.tid = threadIdx.x;
	synthesis_cta<N, ONE>( a, (int64_t) blockIdx.x, env, ola, x0, x1, rowbuf );
	}

// Mirrored first pass (pv_body.cuh: synthesis_cta_mirror): 16 points per thread, thread-private row FIFO and overlap-add ring.
template<int N, int TPS, bool ONE, bool GEN>
__global__ void __launch_bounds__( N / 32, min_blocks( N / 32, TPS ) ) pv_synthesis_mirror_kernel( const SynthArgs a )
	{
	constexpr bool TM = synthesis_uses_tmem<N, TPS, GEN>();
	extern __shared__ __align__( 16 ) unsigned char smem_raw[];
	float2 * ring = TM ? nullptr : reinterpret_cast<float2 *>( smem_raw );  // N/2 pairs (TM: the partials are in tensor memory)
	float2 * x0 = reinterpret_cast<float2 *>( smem_raw ) + ( TM ? 0 : N / 2 );
	float2 * x1 = ONE ? x0 : x0 + XBuf<N / 2>::size;
	float2 * rowbuf = x1 + XBuf<N / 2>::size;                               // N/2 + 2 pairs
	__shared__ __align__( 8 ) DeviceEnv::BulkBarrier bar;
	DeviceEnv env; env.tid = threadIdx.x;
	if constexpr( TM )
		{
		__shared__ uint32_t tmem_slot;
		TmemScope<SY_TM_COLS> scope( &tmem_slot );
		env.tmem = scope.base();
		synthesis_cta_mirror<N, ONE, GEN, true>( a, (int64_t) blockIdx.x, env, ring, x0, x1, rowbuf, &bar );
		}
	else synthesis_cta_mirror<N, ONE, GEN, false>( a, (int64_t) blockIdx.x, env, ring, x0, x1, rowbuf, &bar );
	}

// One thread per (channel, segment, bin): summary of the segment's phase increments.
__global__ void __launch_bounds__( 256 ) pv_phase_seg_kernel( const PhaseSegArgs a )
	{
	const int bchunks = ( a.B + 255 ) / 256;
	const int64_t blk = blockIdx.x;
	const int b = (int)( blk % bchunks ) * 256 + threadIdx.x;
	const int seg = (int)( ( blk / bchunks ) % a.segs_per_channel );
	const int c = (int)( blk / ( (int64_t) bchunks * a.segs_per_channel ) );
	if( b >= a.B ) return;
	const int64_t fa = a.frame_begin + (int64_t) seg * a.seg_len;
	const int64_t fb = ( fa + a.seg_len < a.frame_end ) ? fa + a.seg_len : a.frame_end;
	const float2 * col = a.pv + (int64_t) c * a.pv_channel_stride + ( fa - a.frame_begin ) * (int64_t) a.B + b;
	int flag = 0;
	const PhaseSeg s = phase_segment_summary( col, (int64_t) a.B, fb - fa, a.k, a.P, a.rcpP, flag,
		[]( const float2 * p ) { return __ldg( p ); } );
	PhaseSeg * dst = a.seg_out + ( (int64_t) c * a.segs_per_channel + seg ) * a.B + b;
	*dst = s;
	if( flag ) *a.nan_flag = 1;
	}

// Summaries left by the analysis kernel (analysis_cta<EMIT>): the entries it marked -- always the lowest bins, whose
// expected phase advance is too small for the 32-bit form; every bin of a segment of digital silence, whose frequencies
// are nowhere near their bins' centres; NaN / Inf -- are recomputed from the rows, one thread per (channel, segment, bin),
// all at once: unmarked entries cost a 8-byte read, a fully marked buffer what pv_phase_seg_kernel costs. (The scan's
// group reduction repairs what a caller-limited launch leaves.)
__global__ void __launch_bounds__( 64 ) pv_phase_fix_kernel( const PhaseScanArgs a, int bins )
	{
	const int b = threadIdx.x + blockIdx.z * 64;
	const int s = blockIdx.x, c = blockIdx.y;
	if( b >= bins || b >= a.B ) return;
	PhaseSeg * e = const_cast<PhaseSeg *>( a.seg ) + ( (int64_t) c * a.segs_per_channel + s ) * a.B + b;
	if( !( e->sum.q != e->sum.q ) ) return;
	const int64_t fa = a.fix_frame_begin + (int64_t) s * a.fix_seg_len;
	const int64_t fb = ( fa + a.fix_seg_len < a.fix_frame_end ) ? fa + a.fix_seg_len : a.fix_frame_end;
	const float2 * col = a.fix_pv + (int64_t) c * a.fix_channel_stride + ( fa - a.fix_frame_begin ) * (int64_t) a.B + b;
	int flag = 0;
	*e = phase_segment_summary( col, (int64_t) a.B, fb - fa, a.fix_k, a.P, a.rcpP, flag, []( const float2 * p ) { return __ldg( p ); } );
	if( flag ) *a.fix_nan_flag = 1;
	}

// One thread per (channel, bin): serial walk over the segments (a few thousand at most), writing the
// accumulator value that enters each segment. carry_in/carry_out chain frame-range shards across GPUs.
// The scan over segments runs in three short phases so that its serial depth is group_len + groups + group_len
// instead of segs_per_channel (the combine is associative):
//   mode 0  reduce each group of consecutive segments to one state          thread per (channel, group, bin)
//   mode 1  exclusive scan of the group states (carry_in / carry_out here)  thread per (channel, bin)
//   mode 2  re-walk each group from its prefix, writing acc_start           thread per (channel, group, bin)
__global__ void __launch_bounds__( 128 ) pv_phase_scan_kernel( const PhaseScanArgs a, int mode )
	{
	const int b = blockIdx.x * blockDim.x + threadIdx.x;
	const int g = blockIdx.y;
	const int c = blockIdx.z;
	if( b >= a.B ) return;
	PhaseSeg st; st.sum.q = 0.0; st.sum.r = 0.0; st.mx.q = 0.0; st.mx.r = 0.0;
	PhaseSeg * grp = a.group + (int64_t) c * a.groups * a.B + b;
	if( mode == 1 )
		{
		if( a.carry_in ) st = a.carry_in[(int64_t) c * a.B + b];
		for( int i = 0; i < a.groups; ++i )
			{
			const PhaseSeg tmp = grp[(int64_t) i * a.B];
			grp[(int64_t) i * a.B] = st;
			phase_state_combine( st, tmp, a.P, a.rcpP );
			}
		if( a.carry_out ) a.carry_out[(int64_t) c * a.B + b] = st;
		return;
		}
	const int s0 = g * a.group_len;
	const int s1 = ( s0 + a.group_len < a.segs_per_channel ) ? s0 + a.group_len : a.segs_per_channel;
	const PhaseSeg * src = a.seg + (int64_t) c * a.segs_per_channel * a.B + b;
	if( mode == 0 )
		{
		for( int s = s0; s < s1; ++s )
			{
			PhaseSeg v = src[(int64_t) s * a.B];
			if( a.fix_pv && is_nan_marker( v ) )
				{
				const int64_t fa = a.fix_frame_begin + (int64_t) s * a.fix_seg_len;
				const int64_t fb = ( fa + a.fix_seg_len < a.fix_frame_end ) ? fa + a.fix_seg_len : a.fix_frame_end;
				const float2 * col = a.fix_pv + (int64_t) c * a.fix_channel_stride + ( fa - a.fix_frame_begin ) * (int64_t) a.B + b;
				int flag = 0;
				v = phase_segment_summary( col, (int64_t) a.B, fb - fa, a.fix_k, a.P, a.rcpP, flag, []( const float2 * p ) { return __ldg( p ); } );
				if( flag ) *a.fix_nan_flag = 1;
				const_cast<PhaseSeg *>( src )[(int64_t) s * a.B] = v;
				}
			phase_state_combine( st, v, a.P, a.rcpP );
			}
		grp[(int64_t) g * a.B] = st;
		return;
		}
	st = grp[(int64_t) g * a.B];
	if( a.expand_only && a.expand_carry )
		{
		PhaseSeg cin = a.expand_carry[(int64_t) c * a.B + b];
		phase_state_combine( cin, st, a.P, a.rcpP );
		st = cin;
		}
	double * dst = a.acc_start + (int64_t) c * a.segs_per_channel * a.B + b;
	for( int s = s0; s < s1; ++s )
		{
		dst[(int64_t) s * a.B] = phase_state_value( st, a.P );
		phase_state_combine( st, src[(int64_t) s * a.B], a.P, a.rcpP );
		}
	}

// The same scan for signals of a few hundred segments per channel, where the three launches above are all latency:
// one launch, a CTA per (channel, 32 bins), 16 thread rows that each reduce a contiguous run of segments, one serial
// scan over the 16 run totals in shared memory, then every row re-walks its run from its prefix. Serial depth
// 2 * ceil(segs / 16) + 16 instead of segs.
__global__ void __launch_bounds__( 512 ) pv_phase_scan_small_kernel( const PhaseScanArgs a )
	{
	constexpr int G = 16;
	__shared__ PhaseSeg tot[G][32];
	const int lane = threadIdx.x, g = threadIdx.y;
	const int b = blockIdx.x * 32 + lane;
	const int c = blockIdx.y;
	const bool live = b < a.B;
	const int per = ( a.segs_per_channel + G - 1 ) / G;
	const int s0 = g * per;
	const int s1 = ( s0 + per < a.segs_per_channel ) ? s0 + per : a.segs_per_channel;
	const PhaseSeg * src = a.seg + (int64_t) c * a.segs_per_channel * a.B + b;
	PhaseSeg st; st.sum.q = 0.0; st.sum.r = 0.0; st.mx.q = 0.0; st.mx.r = 0.0;
	if( live ) for( int s = s0; s < s1; ++s ) phase_state_combine( st, src[(int64_t) s * a.B], a.P, a.rcpP );
	tot[g][lane] = st;
	__syncthreads();
	if( g == 0 && live )
		{
		PhaseSeg run; run.sum.q = 0.0; run.sum.r = 0.0; run.mx.q = 0.0; run.mx.r = 0.0;
		if( a.carry_in ) run = a.carry_in[(int64_t) c * a.B + b];
		for( int i = 0; i < G; ++i )
			{
			const PhaseSeg tmp = tot[i][lane];
			tot[i][lane] = run;
			phase_state_combine( run, tmp, a.P, a.rcpP );
			}
		if( a.carry_out ) a.carry_out[(int64_t) c * a.B + b] = run;
		}
	__syncthreads();
	if( !live || !a.acc_start ) return;
	st = tot[g][lane];
	double * dst = a.acc_start + (int64_t) c * a.segs_per_channel * a.B + b;
	for( int s = s0; s < s1; ++s )
		{
		dst[(int64_t) s * a.B] = phase_state_value( st, a.P );
		phase_state_combine( st, src[(int64_t) s * a.B], a.P, a.rcpP );
		}
	}

// carry[r] = summaries[0] (+) ... (+) summaries[r-1], for this rank r.
__global__ void __launch_bounds__( 128 ) pv_phase_carry_kernel( const PhaseSeg * all, int rank, int64_t per_rank, PhaseSeg * carry, double P, double rcpP )
	{
	const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	if( i >= per_rank ) return;
	PhaseSeg st; st.sum.q = 0.0; st.sum.r = 0.0; st.mx.q = 0.0; st.mx.r = 0.0;
	for( int r = 0; r < rank; ++r ) phase_state_combine( st, all[(int64_t) r * per_rank + i], P, rcpP );
	carry[i] = st;
	}

// Audio::convert_to_mid_side (AudioConversions.cpp:42-49): (L +- R) / sqrt(2.0f), IEEE division.
__global__ void __launch_bounds__( 256 ) pv_mid_side_kernel( const float * in, float * out, int64_t n )
	{
	const float sqrt2 = 1.41421356237309504880f;
	for( int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x )
		{
		const float l = in[i], r = in[n + i];
		out[i]     = __fdiv_rn( __fadd_rn( l, r ), sqrt2 );
		out[n + i] = __fdiv_rn( __fsub_rn( l, r ), sqrt2 );
		}
	}

// Clears the output samples the resynthesis kernels reach with red.add (those shared by two segments, and the head and
// tail of the local span) instead of the whole output: every other sample is written exactly once by a plain store.
// Region j of a channel lies between the interior of segment j-1 and the interior of segment j (pv_body.cuh:
// interior_lo = hop*fa + W/2 - hop, interior_hi = hop*fb - W/2; an empty interior counts as the point interior_lo).
// Requires hop <= window (no gaps between the frames' windows).
__global__ void __launch_bounds__( 256 ) pv_zero_shared_kernel( float * out, int64_t out_stride, int64_t out_offset, int64_t out_len,
                                                                 int64_t frame_begin, int64_t frame_end, int seg_len, int segs, int W, int hop )
	{
	const int j = blockIdx.x;            // 0 .. segs
	const int c = blockIdx.y;
	const int half = W / 2;
	auto seg_lo = [&]( int s ) { return (int64_t) hop * ( frame_begin + (int64_t) s * seg_len ) + half - hop; };
	auto seg_hi = [&]( int s )
		{
		const int64_t fa = frame_begin + (int64_t) s * seg_len;
		const int64_t fb = ( fa + seg_len < frame_end ) ? fa + seg_len : frame_end;
		const int64_t hi = (int64_t) hop * fb - half, lo = seg_lo( s );
		return hi > lo ? hi : lo;
		};
	int64_t lo = ( j == 0 ) ? out_offset : seg_hi( j - 1 );
	int64_t hi = ( j == segs ) ? out_offset + out_len : seg_lo( j );
	if( lo < out_offset ) lo = out_offset;
	if( hi > out_offset + out_len ) hi = out_offset + out_len;
	float * dst = out + (int64_t) c * out_stride - out_offset;
	for( int64_t i = lo + threadIdx.x; i < hi; i += blockDim.x ) dst[i] = 0.0f;
	}

cudaError_t launch_zero_shared( float * out, int64_t out_stride, int64_t out_offset, int64_t out_len, int C,
                                int64_t frame_begin, int64_t frame_end, int seg_len, int segs, int W, int hop, cudaStream_t st )
	{
	const dim3 grid( (unsigned)( segs + 1 ), (unsigned) C );
	pv_zero_shared_kernel<<<grid, 256, 0, st>>>( out, out_stride, out_offset, out_len, frame_begin, frame_end, seg_len, segs, W, hop );
	return cudaGetLastError();
	}

// out[i] += add[i] (overlap-add halo received from a neighbouring frame-range shard)
__global__ void __launch_bounds__( 256 ) pv_add_kernel( float * out, const float * add, int64_t n )
	{
	for( int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x )
		out[i] = __fadd_rn( out[i], add[i] );
	}

// ------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------
// Development aids (FLAN_B200_DEBUG builds only): FLAN_B200_SMEM_PAD=<bytes> inflates the dynamic shared memory request
// so that fewer CTAs fit per SM; FLAN_B200_CARVEOUT=<percent> sets the preferred shared-memory carveout of the transforms
// (the 8-point resynthesis excepted).
#ifdef FLAN_B200_DEBUG
static int carveout()
	{
	static const int v = [] { const char * e = std::getenv( "FLAN_B200_CARVEOUT" ); return e ? std::atoi( e ) : -1; }();
	return v;
	}
static void apply_carveout( const void * kernel )
	{
	if( carveout() >= 0 ) cudaFuncSetAttribute( kernel, cudaFuncAttributePreferredSharedMemoryCarveout, carveout() );
	}
static size_t smem_pad()
	{
	static const size_t pad = [] { const char * e = std::getenv( "FLAN_B200_SMEM_PAD" ); return e ? (size_t) std::atol( e ) : (size_t) 0; }();
	return pad;
	}
#else
static void apply_carveout( const void * ) {}
static constexpr size_t smem_pad() { return 0; }
#endif

// CTAs per SM of a kernel that allocates COLS columns of tensor memory. The driver's occupancy query answers 1 for such
// kernels (measured on a B200, tools/micro/tmem.cu: query 1, 4 resident), so the bound is taken from the register file
// and the thread limit, and it must not exceed what the columns allow (512 / COLS): surplus CTAs would wait in
// tcgen05.alloc for others of the same launch to finish. Evaluated once per kernel.
template<auto KERNEL, int THREADS, int COLS> static cudaError_t tmem_kernel_ctas( int * ctas )
	{
	static int n = 0;
	static const cudaError_t r = []
		{
		cudaFuncAttributes fa;
		const cudaError_t e = cudaFuncGetAttributes( &fa, KERNEL );
		if( e != cudaSuccess ) return e;
		const int by_regs = 65536 / ( ( fa.numRegs > 0 ? fa.numRegs : 1 ) * THREADS ), by_threads = 2048 / THREADS;
		n = by_regs < by_threads ? by_regs : by_threads;
		return n * COLS <= 512 ? cudaSuccess : cudaErrorInvalidConfiguration;
		}();
	*ctas = n;
	return r;
	}

// One instantiation of a transform kernel: its descriptor, entry point, threads per CTA, the bytes of one exchange
// buffer, and for the kernels that allocate tensor memory the CTAs per SM that allocation admits.
struct KernelEntry
	{
	TransformKernel k;
	const void * fn;
	int threads;
	size_t xbuf;
	cudaError_t ( *tmem_ctas )( int * );
	};

template<int N, int PT, int TPS, bool ONE, bool PAD, bool EMIT> static KernelEntry analysis_entry()
	{
	constexpr auto fn = pv_analysis_kernel<N, PT, TPS, ONE, PAD, EMIT>;
	return { { KernelKind::analysis, N, PT, TPS, ONE, PAD, EMIT, false }, (const void *) fn, N / ( 2 * PT ), sizeof( float2 ) * XBuf<N / 2>::size,
	         analysis_uses_tmem<N, PT, TPS>() ? &tmem_kernel_ctas<fn, N / ( 2 * PT ), AN_TM_COLS> : nullptr };
	}
template<int N, int TPS> static KernelEntry analysis_mirror_entry()
	{
	return { { KernelKind::analysis_mirror, N, 16, TPS, true, false, false, false }, (const void *) pv_analysis_mirror_kernel<N, TPS>, N / 32,
	         sizeof( float2 ) * XBuf<N / 2>::size, nullptr };
	}
template<int N, int TPS, bool ONE> static KernelEntry synthesis_entry()
	{
	return { { KernelKind::synthesis, N, 8, TPS, ONE, false, false, false }, (const void *) pv_synthesis_kernel<N, TPS, ONE>, N / 16,
	         sizeof( float2 ) * XBuf<N / 2>::size, nullptr };
	}
template<int N, int TPS, bool ONE, bool GEN> static KernelEntry synthesis_mirror_entry()
	{
	constexpr auto fn = pv_synthesis_mirror_kernel<N, TPS, ONE, GEN>;
	return { { KernelKind::synthesis_mirror, N, 16, TPS, ONE, false, false, GEN }, (const void *) fn, N / 32, sizeof( float2 ) * XBuf<N / 2>::size,
	         synthesis_uses_tmem<N, TPS, GEN>() ? &tmem_kernel_ctas<fn, N / 32, SY_TM_COLS> : nullptr };
	}

#ifdef FLAN_B200_DEBUG
// Development builds also carry the register and buffer variants the FLAN_B200_* knobs reach (pv_capi.cu: the knobs of
// analysis_kernel / synthesis_kernel), for the experiments under tools/experiments.
template<int... V, class F> static void each( F && f ) { ( f( std::integral_constant<int, V>() ), ... ); }
template<int N> static void add_variants( std::vector<KernelEntry> & v )
	{
	each<512, 768, 1024>( [&]( auto tps )
		{
		v.push_back( analysis_entry<N, 8, decltype( tps )::value, false, false, false>() );
		v.push_back( synthesis_entry<N, decltype( tps )::value, false>() );
		} );
	if constexpr( N >= 512 )
		each<384, 512, 640, 768>( [&]( auto tps )
			{
			constexpr int TPS = decltype( tps )::value;
			v.push_back( analysis_entry<N, 16, TPS, false, false, false>() );
			v.push_back( analysis_entry<N, 16, TPS, true, false, false>() );
			v.push_back( analysis_entry<N, 16, TPS, true, true, false>() );
			if constexpr( N >= 1024 && N <= 4096 ) v.push_back( analysis_mirror_entry<N, TPS>() );
			} );
	if constexpr( N >= 1024 && N <= 4096 )
		each<384, 512>( [&]( auto tps )
			{
			constexpr int TPS = decltype( tps )::value;
			v.push_back( synthesis_mirror_entry<N, TPS, false, false>() ); v.push_back( synthesis_mirror_entry<N, TPS, false, true>() );
			v.push_back( synthesis_mirror_entry<N, TPS, true, false>() ); v.push_back( synthesis_mirror_entry<N, TPS, true, true>() );
			} );
	if constexpr( N == 8192 ) { v.push_back( synthesis_mirror_entry<N, 256, false, false>() ); v.push_back( synthesis_mirror_entry<N, 256, false, true>() ); }
	}
#endif

// The instantiations of this build: pv_kernel_list.h (development builds: and their variants).
static const std::vector<KernelEntry> & kernels()
	{
	static const std::vector<KernelEntry> list = []
		{
#define PV_A( N, PT, TPS, ONE, PAD, EMIT ) analysis_entry<N, PT, TPS, ONE, PAD, EMIT>(),
#define PV_AM( N, TPS ) analysis_mirror_entry<N, TPS>(),
#define PV_S( N, TPS, ONE ) synthesis_entry<N, TPS, ONE>(),
#define PV_SM( N, TPS, ONE, GEN ) synthesis_mirror_entry<N, TPS, ONE, GEN>(),
		std::vector<KernelEntry> v{ PV_RELEASE_KERNELS( PV_A, PV_AM, PV_S, PV_SM ) };
#undef PV_A
#undef PV_AM
#undef PV_S
#undef PV_SM
#ifdef FLAN_B200_DEBUG
		add_variants<256>( v ); add_variants<512>( v ); add_variants<1024>( v ); add_variants<2048>( v ); add_variants<4096>( v ); add_variants<8192>( v );
#endif
		return v;
		}();
	return list;
	}

// The entry of a descriptor whose kind takes these arguments, or null.
template<class Args> static const KernelEntry * find_kernel( const TransformKernel & k )
	{
	if( k.is_analysis() != std::is_same_v<Args, AnalysisArgs> ) return nullptr;
	for( const KernelEntry & e : kernels() ) if( e.k == k ) return &e;
	return nullptr;
	}

// Dynamic shared memory: the exchange buffers (one when they alias), then the analysis's per-bin sums (EMIT), the
// mirrored analysis's window ring and scratch, or the resynthesis's overlap-add ring and row buffer. The tensor-memory
// kernels keep the per-bin sums and the overlap-add partials in tensor memory instead.
static size_t smem_bytes( const KernelEntry & e, int one_buffer )
	{
	const TransformKernel & k = e.k;
	const bool tm = e.tmem_ctas != nullptr;
	switch( k.kind )
		{
		case KernelKind::analysis: return ( k.ONE ? 1 : 2 ) * e.xbuf + ( k.EMIT && !tm ? sizeof( int ) * ( k.N / 2 + 4 ) : 0 ) + smem_pad();
		case KernelKind::analysis_mirror: return ( one_buffer ? 1 : 2 ) * e.xbuf + sizeof( float2 ) * ( k.N / 2 + 16 ) + smem_pad();
		case KernelKind::synthesis_mirror: return ( tm ? 0 : sizeof( float ) * k.N ) + ( k.ONE ? 1 : 2 ) * e.xbuf + sizeof( float2 ) * ( k.N / 2 + 2 ) + smem_pad();
		default: return sizeof( float ) * k.N + ( k.ONE ? 1 : 2 ) * e.xbuf + sizeof( float2 ) * ( k.N / 2 + 2 ) + smem_pad();
		}
	}

// Sets the kernel's shared-memory size (and in development builds the carveout); a tensor-memory kernel's CTAs per SM
// go to *tmem_ctas (0 for the others).
static cudaError_t prepare( const KernelEntry & e, size_t smem, int * tmem_ctas )
	{
	*tmem_ctas = 0;
	const cudaError_t r = cudaFuncSetAttribute( e.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem );
	if( r != cudaSuccess ) return r;
	if( e.k.kind != KernelKind::synthesis ) apply_carveout( e.fn );
	return e.tmem_ctas ? e.tmem_ctas( tmem_ctas ) : cudaSuccess;
	}

template<class Args> static cudaError_t launch_kernel( const TransformKernel & k, const Args & a, int64_t blocks, cudaStream_t st )
	{
	const KernelEntry * e = find_kernel<Args>( k );
	if( !e ) return cudaErrorInvalidValue;
	const size_t smem = smem_bytes( *e, a.one_buffer );
	int ctas = 0;
	const cudaError_t r = prepare( *e, smem, &ctas );
	if( r != cudaSuccess ) return r;
	void * args[] = { const_cast<Args *>( &a ) };
	cudaLaunchKernel( e->fn, dim3( (unsigned) blocks ), dim3( (unsigned) e->threads ), args, smem, st );
	return cudaGetLastError();
	}

template<class Args> static cudaError_t kernel_ctas( const TransformKernel & k, const Args & a, int * ctas )
	{
	*ctas = 0;
	const KernelEntry * e = find_kernel<Args>( k );
	if( !e ) return cudaErrorInvalidValue;
	const size_t smem = smem_bytes( *e, a.one_buffer );
	const cudaError_t r = prepare( *e, smem, ctas );
	if( r != cudaSuccess || e->tmem_ctas ) return r;
	return cudaOccupancyMaxActiveBlocksPerMultiprocessor( ctas, e->fn, e->threads, smem );
	}

cudaError_t launch( const TransformKernel & k, const AnalysisArgs & a, int64_t blocks, cudaStream_t st ) { return launch_kernel( k, a, blocks, st ); }
cudaError_t launch( const TransformKernel & k, const SynthArgs & a, int64_t blocks, cudaStream_t st ) { return launch_kernel( k, a, blocks, st ); }
cudaError_t resident_ctas( const TransformKernel & k, const AnalysisArgs & a, int * ctas ) { return kernel_ctas( k, a, ctas ); }
cudaError_t resident_ctas( const TransformKernel & k, const SynthArgs & a, int * ctas ) { return kernel_ctas( k, a, ctas ); }

cudaError_t launch_phase_seg( const PhaseSegArgs & a, int C, cudaStream_t st )
	{
	const int64_t blocks = (int64_t)( ( a.B + 255 ) / 256 ) * a.segs_per_channel * C;
	pv_phase_seg_kernel<<<(unsigned) blocks, 256, 0, st>>>( a );
	return cudaGetLastError();
	}

cudaError_t launch_phase_scan( const PhaseScanArgs & a, int C, cudaStream_t st )
	{
	const dim3 wide( ( a.B + 127 ) / 128, a.groups, C ), narrow( ( a.B + 127 ) / 128, 1, C );
	if( a.segs_per_channel <= 256 && C <= 65535 && !a.expand_only )     // latency-bound sizes: one launch instead of three
		{
		pv_phase_scan_small_kernel<<<dim3( ( a.B + 31 ) / 32, C ), dim3( 32, 16 ), 0, st>>>( a );
		return cudaGetLastError();
		}
	if( !a.expand_only )
		{
		if( a.fix_pv && C <= 65535 && ( a.B + 63 ) / 64 <= 65535 )
			pv_phase_fix_kernel<<<dim3( a.segs_per_channel, C, ( a.B + 63 ) / 64 ), 64, 0, st>>>( a, a.B );
		pv_phase_scan_kernel<<<wide, 128, 0, st>>>( a, 0 );
		pv_phase_scan_kernel<<<narrow, 128, 0, st>>>( a, 1 );
		}
	if( a.acc_start ) pv_phase_scan_kernel<<<wide, 128, 0, st>>>( a, 2 );
	return cudaGetLastError();
	}

cudaError_t launch_phase_carry( const PhaseSeg * all, int rank, int64_t per_rank, PhaseSeg * carry, double P, double rcpP, cudaStream_t st )
	{
	pv_phase_carry_kernel<<<(unsigned)( ( per_rank + 127 ) / 128 ), 128, 0, st>>>( all, rank, per_rank, carry, P, rcpP );
	return cudaGetLastError();
	}

cudaError_t launch_mid_side( const float * in, float * out, int64_t n, int sms, cudaStream_t st )
	{
	int64_t blocks = ( n + 255 ) / 256;
	if( blocks > (int64_t) sms * 16 ) blocks = (int64_t) sms * 16;
	if( blocks < 1 ) blocks = 1;
	pv_mid_side_kernel<<<(unsigned) blocks, 256, 0, st>>>( in, out, n );
	return cudaGetLastError();
	}

cudaError_t launch_add( float * out, const float * add, int64_t n, int sms, cudaStream_t st )
	{
	int64_t blocks = ( n + 255 ) / 256;
	if( blocks > (int64_t) sms * 16 ) blocks = (int64_t) sms * 16;
	if( blocks < 1 ) blocks = 1;
	pv_add_kernel<<<(unsigned) blocks, 256, 0, st>>>( out, add, n );
	return cudaGetLastError();
	}


__global__ void __launch_bounds__( 1024 ) pv_state_push_kernel( const StatePush p )
	{
	uint4 * dst = p.dst[blockIdx.x];
	for( unsigned i = threadIdx.x; i < p.n16; i += blockDim.x ) dst[i] = p.src[i];
	__threadfence_system();
	__syncthreads();
	if( threadIdx.x == 0 && p.count[blockIdx.x] )
		{
		__threadfence_system();
		atomicAdd_system( p.count[blockIdx.x], 1u );      // the destination waits for ONE value: (its rank) x (steps of this parity)
		}
	}

cudaError_t launch_state_push( const StatePush & p, int destinations, cudaStream_t st )
	{
	if( destinations < 1 ) return cudaSuccess;
	if( destinations > 16 ) return cudaErrorInvalidValue;
	pv_state_push_kernel<<<destinations, 1024, 0, st>>>( p );
	return cudaGetLastError();
	}

} // namespace pvk
