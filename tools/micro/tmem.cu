// Tensor memory (TMEM) used as per-thread storage, no MMA: dependent-chain latency of tcgen05.ld.32x32b.x{4,16,32} +
// tcgen05.wait::ld against an L1-hit LDG.64 and an LDS.64, and per-SM load throughput with 16 resident warps
// (4 CTAs x 128 threads, 128 columns each: the whole 512-column TMEM of the SM); tcgen05.st.32x32b.x8 throughput alone
// and interleaved with loads, and the latency of a store -> wait::st -> load round trip on one column.
//
//     nvcc -std=c++17 -O3 -gencode arch=compute_100a,code=sm_100a -o tools/micro/tmem.bin tools/micro/tmem.cu
#include <cstdio>
#include <cstdint>
#include <cuda_runtime.h>

#define CK( x ) do { cudaError_t e_ = ( x ); if( e_ != cudaSuccess ) { printf( "%s: %s\n", #x, cudaGetErrorString( e_ ) ); return 1; } } while( 0 )

constexpr int COLS = 128, ITERS = 2048;

__device__ __forceinline__ uint32_t tm_alloc( uint32_t * slot )
	{
	if( threadIdx.x < 32 )
		{
		asm volatile( "tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"( (unsigned) __cvta_generic_to_shared( slot ) ), "n"( COLS ) : "memory" );
		asm volatile( "tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory" );
		}
	asm volatile( "tcgen05.fence::before_thread_sync;" ::: "memory" );
	__syncthreads();
	asm volatile( "tcgen05.fence::after_thread_sync;" ::: "memory" );
	return *slot + ( ( threadIdx.x & 96u ) << 16 );         // lane quarter of this warp
	}
__device__ __forceinline__ void tm_free( uint32_t base )
	{
	asm volatile( "tcgen05.fence::before_thread_sync;" ::: "memory" );
	__syncthreads();
	asm volatile( "tcgen05.fence::after_thread_sync;" ::: "memory" );
	if( threadIdx.x < 32 ) asm volatile( "tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"( base ), "n"( COLS ) : "memory" );
	}
__device__ __forceinline__ void tm_st4( uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w )
	{
	asm volatile( "tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" :: "r"( a ), "r"( x ), "r"( y ), "r"( z ), "r"( w ) : "memory" );
	}
__device__ __forceinline__ void tm_wait() { asm volatile( "tcgen05.wait::ld.sync.aligned;" ::: "memory" ); }

// X words from column c; returns their sum's low bits folded into a column index for the next load (dependent chain)
template<int X> __device__ __forceinline__ uint32_t tm_ld_chain( uint32_t a )
	{
	uint32_t r[32];
	if constexpr( X == 4 )
		asm volatile( "tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];" : "=r"( r[0] ), "=r"( r[1] ), "=r"( r[2] ), "=r"( r[3] ) : "r"( a ) : "memory" );
	if constexpr( X == 16 )
		asm volatile( "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
		              : "=r"( r[0] ), "=r"( r[1] ), "=r"( r[2] ), "=r"( r[3] ), "=r"( r[4] ), "=r"( r[5] ), "=r"( r[6] ), "=r"( r[7] ),
		                "=r"( r[8] ), "=r"( r[9] ), "=r"( r[10] ), "=r"( r[11] ), "=r"( r[12] ), "=r"( r[13] ), "=r"( r[14] ), "=r"( r[15] ) : "r"( a ) : "memory" );
	if constexpr( X == 32 )
		asm volatile( "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
		              : "=r"( r[0] ), "=r"( r[1] ), "=r"( r[2] ), "=r"( r[3] ), "=r"( r[4] ), "=r"( r[5] ), "=r"( r[6] ), "=r"( r[7] ),
		                "=r"( r[8] ), "=r"( r[9] ), "=r"( r[10] ), "=r"( r[11] ), "=r"( r[12] ), "=r"( r[13] ), "=r"( r[14] ), "=r"( r[15] ),
		                "=r"( r[16] ), "=r"( r[17] ), "=r"( r[18] ), "=r"( r[19] ), "=r"( r[20] ), "=r"( r[21] ), "=r"( r[22] ), "=r"( r[23] ),
		                "=r"( r[24] ), "=r"( r[25] ), "=r"( r[26] ), "=r"( r[27] ), "=r"( r[28] ), "=r"( r[29] ), "=r"( r[30] ), "=r"( r[31] ) : "r"( a ) : "memory" );
	tm_wait();
	uint32_t s = 0;
#pragma unroll
	for( int i = 0; i < X; ++i ) s += r[i];
	return s;
	}

// Column j holds 0 everywhere, so every chained address is the same column 0 (+0): the load depends on the previous one.
template<int X> __global__ void __launch_bounds__( 128 ) lat_tmem( long long * cyc, uint32_t * sink )
	{
	__shared__ uint32_t slot;
	const uint32_t base = tm_alloc( &slot );
	for( int c = 0; c < COLS; c += 4 ) tm_st4( base + c, 0, 0, 0, 0 );
	asm volatile( "tcgen05.wait::st.sync.aligned;" ::: "memory" );
	uint32_t col = 0;
	col += tm_ld_chain<X>( base + col );           // warm
	const long long t0 = clock64();
#pragma unroll 1
	for( int i = 0; i < ITERS; ++i ) col = tm_ld_chain<X>( base + ( col & 0x60u ) );
	const long long t1 = clock64();
	if( threadIdx.x == 0 ) cyc[0] = t1 - t0;
	sink[threadIdx.x] = col;
	tm_free( slot );
	}

// Pointer chase over 128 float2 that stay in L1 (LDG.64 through the non-coherent path) or in shared memory (LDS.64).
__global__ void __launch_bounds__( 128 ) lat_ldg( const float2 * tab, long long * cyc, uint32_t * sink )
	{
	uint32_t i = threadIdx.x & 127u;
	for( int k = 0; k < 64; ++k ) i = (uint32_t) __ldg( tab + i ).x;         // warm L1
	const long long t0 = clock64();
#pragma unroll 1
	for( int k = 0; k < ITERS; ++k ) i = (uint32_t) __ldg( tab + i ).x;
	const long long t1 = clock64();
	if( threadIdx.x == 0 ) cyc[0] = t1 - t0;
	sink[threadIdx.x] = i;
	}
__global__ void __launch_bounds__( 128 ) lat_lds( const float2 * tab, long long * cyc, uint32_t * sink )
	{
	__shared__ float2 s[128];
	s[threadIdx.x] = tab[threadIdx.x];
	__syncthreads();
	uint32_t i = threadIdx.x & 127u;
	const long long t0 = clock64();
#pragma unroll 1
	for( int k = 0; k < ITERS; ++k ) i = (uint32_t) s[i].x;
	const long long t1 = clock64();
	if( threadIdx.x == 0 ) cyc[0] = t1 - t0;
	sink[threadIdx.x] = i;
	}

// Throughput: every thread reads 16 words per iteration (four independent x4 loads, one wait), 4 CTAs per SM.
__global__ void __launch_bounds__( 128, 4 ) thr_tmem( uint32_t * sink, int iters )
	{
	__shared__ uint32_t slot;
	const uint32_t base = tm_alloc( &slot );
	for( int c = 0; c < COLS; c += 4 ) tm_st4( base + c, c, c + 1, c + 2, c + 3 );
	asm volatile( "tcgen05.wait::st.sync.aligned;" ::: "memory" );
	uint32_t s = 0;
#pragma unroll 1
	for( int i = 0; i < iters; ++i )
		{
		uint32_t r[16];
		const uint32_t a = base + ( ( i * 16 ) & ( COLS - 1 ) );
		asm volatile( "tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];" : "=r"( r[0] ), "=r"( r[1] ), "=r"( r[2] ), "=r"( r[3] ) : "r"( a ) : "memory" );
		asm volatile( "tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];" : "=r"( r[4] ), "=r"( r[5] ), "=r"( r[6] ), "=r"( r[7] ) : "r"( a + 4 ) : "memory" );
		asm volatile( "tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];" : "=r"( r[8] ), "=r"( r[9] ), "=r"( r[10] ), "=r"( r[11] ) : "r"( a + 8 ) : "memory" );
		asm volatile( "tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];" : "=r"( r[12] ), "=r"( r[13] ), "=r"( r[14] ), "=r"( r[15] ) : "r"( a + 12 ) : "memory" );
		tm_wait();
#pragma unroll
		for( int j = 0; j < 16; ++j ) s ^= r[j];
		}
	sink[blockIdx.x * 128 + threadIdx.x] = s;
	tm_free( slot );
	}
// Store throughput: every thread writes 16 words per iteration (two x8 stores), and with LD also reads 16 other words
// (two x8 loads) of the same iteration, one wait::st per iteration either way, 4 CTAs per SM.
template<bool LD> __global__ void __launch_bounds__( 128, 4 ) thr_tmem_st( uint32_t * sink, int iters )
	{
	__shared__ uint32_t slot;
	const uint32_t base = tm_alloc( &slot );
	for( int c = 0; c < COLS; c += 4 ) tm_st4( base + c, c, c + 1, c + 2, c + 3 );
	asm volatile( "tcgen05.wait::st.sync.aligned;" ::: "memory" );
	uint32_t s = threadIdx.x;
#pragma unroll 1
	for( int i = 0; i < iters; ++i )
		{
		const uint32_t a = base + ( ( i * 32 ) & ( COLS - 1 ) );
		const uint32_t v = s + i;
		asm volatile( "tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%1,%1,%1,%1,%1,%1,%1};" :: "r"( a ), "r"( v ) : "memory" );
		asm volatile( "tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%1,%1,%1,%1,%1,%1,%1};" :: "r"( a + 8 ), "r"( v ) : "memory" );
		if( LD )
			{
			uint32_t r[16];
			asm volatile( "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
			              : "=r"( r[0] ), "=r"( r[1] ), "=r"( r[2] ), "=r"( r[3] ), "=r"( r[4] ), "=r"( r[5] ), "=r"( r[6] ), "=r"( r[7] ) : "r"( a + 16 ) : "memory" );
			asm volatile( "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
			              : "=r"( r[8] ), "=r"( r[9] ), "=r"( r[10] ), "=r"( r[11] ), "=r"( r[12] ), "=r"( r[13] ), "=r"( r[14] ), "=r"( r[15] ) : "r"( a + 24 ) : "memory" );
			tm_wait();
#pragma unroll
			for( int j = 0; j < 16; ++j ) s ^= r[j];
			}
		asm volatile( "tcgen05.wait::st.sync.aligned;" ::: "memory" );
		}
	sink[blockIdx.x * 128 + threadIdx.x] = s;
	tm_free( slot );
	}

// Round trip on one column: x2 store, wait::st, x2 load of the same column, wait::ld; the loaded value feeds the next
// store (dependent chain).
__global__ void __launch_bounds__( 128 ) lat_tmem_rt( long long * cyc, uint32_t * sink )
	{
	__shared__ uint32_t slot;
	const uint32_t base = tm_alloc( &slot );
	uint32_t x = threadIdx.x, y = 0;
	long long t0 = 0;
#pragma unroll 1
	for( int i = -1; i < ITERS; ++i )
		{
		if( i == 0 ) t0 = clock64();
		asm volatile( "tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1,%2};" :: "r"( base + 96 ), "r"( x ), "r"( y ) : "memory" );
		asm volatile( "tcgen05.wait::st.sync.aligned;" ::: "memory" );
		asm volatile( "tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0,%1}, [%2];" : "=r"( x ), "=r"( y ) : "r"( base + 96 ) : "memory" );
		tm_wait();
		x += 1u;
		}
	const long long t1 = clock64();
	if( threadIdx.x == 0 ) cyc[0] = t1 - t0;
	sink[threadIdx.x] = x + y;
	tm_free( slot );
	}

// The same 16 words per thread per iteration as eight LDG.64 from a 2 KB table (L1 hits), 4 CTAs per SM.
__global__ void __launch_bounds__( 128, 4 ) thr_ldg( const float2 * tab, uint32_t * sink, int iters )
	{
	uint32_t s = 0;
	const int t = threadIdx.x;
#pragma unroll 1
	for( int i = 0; i < iters; ++i )
		{
#pragma unroll
		for( int j = 0; j < 8; ++j )
			{
			const float2 v = __ldg( tab + ( ( t + j * 16 + i ) & 255 ) );
			s ^= __float_as_uint( v.x ) ^ __float_as_uint( v.y );
			}
		}
	sink[blockIdx.x * 128 + threadIdx.x] = s;
	}

// Residency: the most CTAs of one launch that were on one SM at the same time (each CTA stays ~20 us), for a kernel
// that allocates 128 columns and for the same kernel without tensor memory.
template<bool TM> __global__ void __launch_bounds__( 128, 4 ) resident( unsigned * active, unsigned * peak )
	{
	__shared__ uint32_t slot;
	uint32_t base = 0;
	if( TM ) base = tm_alloc( &slot );
	unsigned sm;
	asm volatile( "mov.u32 %0, %%smid;" : "=r"( sm ) );
	if( threadIdx.x == 0 ) { const unsigned n = atomicAdd( active + sm, 1u ) + 1u; atomicMax( peak + sm, n ); }
	const long long t0 = clock64();
	while( clock64() - t0 < 40000 ) {}
	__syncthreads();
	if( threadIdx.x == 0 ) atomicSub( active + sm, 1u );
	if( TM ) tm_free( slot );
	(void) base;
	}

int main()
	{
	cudaDeviceProp prop;
	CK( cudaGetDeviceProperties( &prop, 0 ) );
	int clk_khz = 0;
	CK( cudaDeviceGetAttribute( &clk_khz, cudaDevAttrClockRate, 0 ) );
	printf( "device: %s, %d SMs, max SM clock %d MHz\n", prop.name, prop.multiProcessorCount, clk_khz / 1000 );
	float2 * tab; long long * cyc; uint32_t * sink;
	CK( cudaMalloc( &tab, 256 * sizeof( float2 ) ) );
	CK( cudaMalloc( &cyc, sizeof( long long ) ) );
	CK( cudaMalloc( &sink, (size_t) prop.multiProcessorCount * 4 * 128 * sizeof( uint32_t ) ) );
	float2 h[256];
	for( int i = 0; i < 256; ++i ) { h[i].x = (float)( ( i * 37 + 11 ) & 127 ); h[i].y = 0.0f; }   // a full-cycle permutation of 0..127
	CK( cudaMemcpy( tab, h, sizeof( h ), cudaMemcpyHostToDevice ) );
	long long c = 0;
	auto lat = [&]( const char * name )
		{
		cudaMemcpy( &c, cyc, sizeof( c ), cudaMemcpyDeviceToHost );
		printf( "latency %-38s %7.1f cycles\n", name, (double) c / ITERS );
		};
	for( int rep = 0; rep < 2; ++rep )
		{
		lat_ldg<<<1, 128>>>( tab, cyc, sink ); CK( cudaDeviceSynchronize() ); lat( "LDG.64 (L1 hit) dependent chain" );
		lat_lds<<<1, 128>>>( tab, cyc, sink ); CK( cudaDeviceSynchronize() ); lat( "LDS.64 dependent chain" );
		lat_tmem<4><<<1, 128>>>( cyc, sink ); CK( cudaDeviceSynchronize() ); lat( "tcgen05.ld.32x32b.x4 + wait::ld" );
		lat_tmem<16><<<1, 128>>>( cyc, sink ); CK( cudaDeviceSynchronize() ); lat( "tcgen05.ld.32x32b.x16 + wait::ld" );
		lat_tmem<32><<<1, 128>>>( cyc, sink ); CK( cudaDeviceSynchronize() ); lat( "tcgen05.ld.32x32b.x32 + wait::ld" );
		lat_tmem_rt<<<1, 128>>>( cyc, sink ); CK( cudaDeviceSynchronize() ); lat( "st.x2 + wait::st + ld.x2 + wait::ld" );
		}
	const int ctas = prop.multiProcessorCount * 4, iters = 1 << 16;
	int occ = 0;
	CK( cudaOccupancyMaxActiveBlocksPerMultiprocessor( &occ, thr_tmem, 128, 0 ) );
	printf( "thr_tmem resident CTAs/SM: %d\n", occ );
	cudaEvent_t e0, e1;
	cudaEventCreate( &e0 ); cudaEventCreate( &e1 );
	auto thr = [&]( const char * name, auto launch )
		{
		launch();
		cudaEventRecord( e0 );
		launch();
		cudaEventRecord( e1 );
		cudaEventSynchronize( e1 );
		float ms = 0.0f;
		cudaEventElapsedTime( &ms, e0, e1 );
		const double bytes = (double) ctas * 128 * iters * 16 * 4;
		printf( "throughput %-34s %8.3f ms  %7.1f B/clk/SM (at max clock)  %s\n", name, ms,
		        bytes / prop.multiProcessorCount / ( ms * 1e-3 * clk_khz * 1e3 ), cudaGetErrorString( cudaGetLastError() ) );
		};
	thr( "TMEM 4 x ld.x4 + wait, 16 warps/SM", [&] { thr_tmem<<<ctas, 128>>>( sink, iters ); } );
	thr( "LDG.64 L1 hits, 16 warps/SM", [&] { thr_ldg<<<ctas, 128>>>( tab, sink, iters ); } );
	thr( "TMEM 2 x st.x8 + wait::st", [&] { thr_tmem_st<false><<<ctas, 128>>>( sink, iters ); } );
	thr( "TMEM 2 x st.x8 + 2 x ld.x8, both waits", [&] { thr_tmem_st<true><<<ctas, 128>>>( sink, iters ); } );
	CK( cudaDeviceSynchronize() );
	unsigned * cnt;
	CK( cudaMalloc( &cnt, 2 * 1024 * sizeof( unsigned ) ) );
	for( int tm = 0; tm < 2; ++tm )
		{
		CK( cudaMemset( cnt, 0, 2 * 1024 * sizeof( unsigned ) ) );
		int q = 0;
		CK( cudaOccupancyMaxActiveBlocksPerMultiprocessor( &q, tm ? resident<true> : resident<false>, 128, 0 ) );
		if( tm ) resident<true><<<prop.multiProcessorCount * 8, 128>>>( cnt, cnt + 1024 );
		else resident<false><<<prop.multiProcessorCount * 8, 128>>>( cnt, cnt + 1024 );
		CK( cudaDeviceSynchronize() );
		unsigned pk[1024];
		CK( cudaMemcpy( pk, cnt + 1024, sizeof( pk ), cudaMemcpyDeviceToHost ) );
		unsigned mx = 0, mn = ~0u;
		for( int i = 0; i < prop.multiProcessorCount; ++i ) { mx = pk[i] > mx ? pk[i] : mx; mn = pk[i] < mn ? pk[i] : mn; }
		printf( "residency %-12s occupancy query %d CTAs/SM, measured peak %u..%u CTAs/SM\n", tm ? "with TMEM" : "without TMEM", q, mn, mx );
		}
	return 0;
	}
