// flan_b200/csrc/pv_io.cu -- sm_100a kernels for the sample codecs of the file formats either side of the path:
//   * .flan RIFF-PV: magnitude / dft size and frequency / sample rate, clamped to [-1,1], times 2^23, truncated, three
//     little-endian bytes each (PVBuffer::save, reference PV/PVBuffer.cpp:99-127; load :253-268);
//   * WAV as the reference writes it through libsndfile (Audio/AudioBuffer.cpp:136-170): clamp, interleave, convert to
//     the file's sample type; and reads it (:112-125): convert to float, de-interleave. The sample types are libsndfile's
//     for SF_FORMAT_WAV -- PCM_U8, PCM_16, PCM_24, PCM_32, FLOAT, DOUBLE -- with its default conversions (normalisation
//     on, clipping off; pcm.c, float32.c, double64.c), restated in struct Pcm below.
// Byte work, HBM-bound: a thread converts four values into as many 32-bit words as one value has bytes (or back); words
// pass through a shared-memory tile so that global traffic on the byte side is full 16-byte vectors.
#include "pv_io.h"

#include "../../include/flan_b200.h"

namespace pvio {

constexpr int THREADS = 256;
constexpr int TILE_VALUES = THREADS * 4;            // values per tile: four a thread, so a thread's bytes are whole words

__device__ __forceinline__ int flan_quantise( float v, float div )
	{
	float x = v / div;                                                  // PVBuffer.cpp:112-113
	x = x < -1.0f ? -1.0f : ( 1.0f < x ? 1.0f : x );                    // std::clamp (NaN passes through)
	const double scaled = (double) x * 8388608.0;
	return ( scaled != scaled ) ? (int) 0x80000000u : (int) scaled;     // truncation; NaN as the x86 conversion gives it
	}

__device__ __forceinline__ void pack4( const int q[4], unsigned w[3] )
	{
	const unsigned a = q[0] & 0xFFFFFF, b = q[1] & 0xFFFFFF, c = q[2] & 0xFFFFFF, d = q[3] & 0xFFFFFF;
	w[0] = a | ( b << 24 );
	w[1] = ( b >> 8 ) | ( c << 16 );
	w[2] = ( c >> 16 ) | ( d << 8 );
	}

__device__ __forceinline__ void unpack4( const unsigned w[3], int q[4] )
	{
	const unsigned a = w[0] & 0xFFFFFF, b = ( w[0] >> 24 ) | ( ( w[1] & 0xFFFF ) << 8 ),
	               c = ( w[1] >> 16 ) | ( ( w[2] & 0xFF ) << 16 ), d = w[2] >> 8;
	const unsigned v[4] = { a, b, c, d };
#pragma unroll
	for( int i = 0; i < 4; ++i ) q[i] = (int)( v[i] << 8 ) >> 8;         // sign-extend 24 -> 32 (PVBuffer.cpp:261)
	}

// A thread's W words in the tile: the widest shared-memory access their alignment (4 * W bytes) allows.
template<int W> __device__ __forceinline__ void put_words( unsigned * tile, const unsigned w[W] )
	{
	unsigned * p = tile + W * threadIdx.x;
	if constexpr( W == 2 ) *reinterpret_cast<uint2 *>( p ) = make_uint2( w[0], w[1] );
	else if constexpr( W % 4 == 0 )
		{
#pragma unroll
		for( int k = 0; k < W; k += 4 ) reinterpret_cast<uint4 *>( p )[k / 4] = make_uint4( w[k], w[k + 1], w[k + 2], w[k + 3] );
		}
	else
		{
#pragma unroll
		for( int k = 0; k < W; ++k ) p[k] = w[k];
		}
	}

template<int W> __device__ __forceinline__ void get_words( const unsigned * tile, unsigned w[W] )
	{
	const unsigned * p = tile + W * threadIdx.x;
	if constexpr( W == 2 ) { const uint2 u = *reinterpret_cast<const uint2 *>( p ); w[0] = u.x; w[1] = u.y; }
	else if constexpr( W % 4 == 0 )
		{
#pragma unroll
		for( int k = 0; k < W; k += 4 )
			{ const uint4 u = reinterpret_cast<const uint4 *>( p )[k / 4]; w[k] = u.x; w[k + 1] = u.y; w[k + 2] = u.z; w[k + 3] = u.w; }
		}
	else
		{
#pragma unroll
		for( int k = 0; k < W; ++k ) w[k] = p[k];
		}
	}

// Tile of THREADS * W words -> global bytes. Full tiles go out as uint4; the last, partial tile byte by byte.
template<int W> __device__ __forceinline__ void store_tile( const unsigned * tile, uint8_t * bytes, int64_t tile_index, int64_t total_bytes )
	{
	constexpr int TILE_BYTES = THREADS * W * 4;
	const int64_t base = tile_index * TILE_BYTES;
	if( base + TILE_BYTES <= total_bytes )
		{
#pragma unroll
		for( int i = threadIdx.x; i < TILE_BYTES / 16; i += THREADS )
			__stcs( reinterpret_cast<uint4 *>( bytes + base ) + i, reinterpret_cast<const uint4 *>( tile )[i] );
		}
	else
		for( int64_t b = threadIdx.x; base + b < total_bytes; b += THREADS )
			bytes[base + b] = (uint8_t)( tile[b >> 2] >> ( 8 * ( b & 3 ) ) );
	}

template<int W> __device__ __forceinline__ void load_tile( unsigned * tile, const uint8_t * bytes, int64_t tile_index, int64_t total_bytes )
	{
	constexpr int TILE_BYTES = THREADS * W * 4;
	const int64_t base = tile_index * TILE_BYTES;
	if( base + TILE_BYTES <= total_bytes )
		{
#pragma unroll
		for( int i = threadIdx.x; i < TILE_BYTES / 16; i += THREADS )
			reinterpret_cast<uint4 *>( tile )[i] = __ldcs( reinterpret_cast<const uint4 *>( bytes + base ) + i );
		}
	else
		{
		for( int w = threadIdx.x; w < THREADS * W; w += THREADS ) tile[w] = 0;
		__syncthreads();
		for( int64_t b = threadIdx.x; base + b < total_bytes; b += THREADS )
			atomicOr( &tile[b >> 2], (unsigned) bytes[base + b] << ( 8 * ( b & 3 ) ) );
		}
	}

// values = 2 * count floats (m, f, m, f, ...); even positions are scaled by the dft size, odd ones by the sample rate.
__global__ void __launch_bounds__( THREADS ) pv_flan_encode_kernel( const float * pv, int64_t values, float dft_size, float sample_rate, uint8_t * bytes )
	{
	__shared__ __align__( 16 ) unsigned tile[THREADS * 3];
	const int64_t tiles = ( values + TILE_VALUES - 1 ) / TILE_VALUES;
	for( int64_t t = blockIdx.x; t < tiles; t += gridDim.x )
		{
		const int64_t v0 = t * TILE_VALUES + 4 * threadIdx.x;
		int q[4] = { 0, 0, 0, 0 };
		if( v0 + 4 <= values )
			{
			const float4 x = __ldcs( reinterpret_cast<const float4 *>( pv + v0 ) );
			q[0] = flan_quantise( x.x, dft_size ); q[1] = flan_quantise( x.y, sample_rate );
			q[2] = flan_quantise( x.z, dft_size ); q[3] = flan_quantise( x.w, sample_rate );
			}
		else
			for( int i = 0; i < 4; ++i ) if( v0 + i < values ) q[i] = flan_quantise( pv[v0 + i], ( i & 1 ) ? sample_rate : dft_size );
		unsigned w[3];
		pack4( q, w );
		put_words<3>( tile, w );
		__syncthreads();
		store_tile<3>( tile, bytes, t, values * 3 );
		__syncthreads();
		}
	}

__global__ void __launch_bounds__( THREADS ) pv_flan_decode_kernel( const uint8_t * bytes, int64_t values, float dft_size, float sample_rate, float * pv )
	{
	__shared__ __align__( 16 ) unsigned tile[THREADS * 3];
	const int64_t tiles = ( values + TILE_VALUES - 1 ) / TILE_VALUES;
	for( int64_t t = blockIdx.x; t < tiles; t += gridDim.x )
		{
		load_tile<3>( tile, bytes, t, values * 3 );
		__syncthreads();
		unsigned w[3];
		get_words<3>( tile, w );
		int q[4];
		unpack4( w, q );
		const int64_t v0 = t * TILE_VALUES + 4 * threadIdx.x;
		float x[4];
#pragma unroll
		for( int i = 0; i < 4; ++i ) x[i] = (float)( (double) q[i] / 8388608.0 ) * ( ( i & 1 ) ? sample_rate : dft_size );   // PVBuffer.cpp:262
		if( v0 + 4 <= values ) __stcs( reinterpret_cast<float4 *>( pv + v0 ), make_float4( x[0], x[1], x[2], x[3] ) );
		else for( int i = 0; i < 4; ++i ) if( v0 + i < values ) pv[v0 + i] = x[i];
		__syncthreads();
		}
	}

// ---- WAV sample types -----------------------------------------------------------------------------------------------
// Pcm<T>: BYTES per value, and four values <-> BYTES little-endian words. Write side: clamp (AudioBuffer.cpp:158-161,
// NaN passes through), then libsndfile's conversion; lrintf is __float2int_rn of a __fmul_rn product (round half to
// even, never contracted). Read side: libsndfile's normalised conversion to float.

__device__ __forceinline__ float clamp1( float s ) { return s < -1.0f ? -1.0f : ( 1.0f < s ? 1.0f : s ); }

template<int T> struct Pcm;

template<> struct Pcm<FLAN_B200_WAV_PCM_U8>
	{
	static constexpr int BYTES = 1;
	// pcm.c f2uc_array: lrintf( x * 0x7F ) + 128. A NaN converts to 0 here and to INT_MIN on x86: either way the low
	// byte of the sum is 128.
	static __device__ __forceinline__ void encode( const float x[4], unsigned w[1] )
		{
		w[0] = 0;
#pragma unroll
		for( int i = 0; i < 4; ++i ) w[0] |= (unsigned)( ( __float2int_rn( __fmul_rn( clamp1( x[i] ), 127.0f ) ) + 128 ) & 0xFF ) << ( 8 * i );
		}
	// pcm.c uc2f_array: ( v - 128 ) * ( 1 / 0x80 )
	static __device__ __forceinline__ void decode( const unsigned w[1], float x[4] )
		{
#pragma unroll
		for( int i = 0; i < 4; ++i ) x[i] = __fmul_rn( (float)( (int)( ( w[0] >> ( 8 * i ) ) & 0xFF ) - 128 ), 1.0f / 128.0f );
		}
	};

template<> struct Pcm<FLAN_B200_WAV_PCM_16>
	{
	static constexpr int BYTES = 2;
	// pcm.c f2les_array: lrintf( x * 0x7FFF ), low two bytes
	static __device__ __forceinline__ void encode( const float x[4], unsigned w[2] )
		{
		unsigned q[4];
#pragma unroll
		for( int i = 0; i < 4; ++i ) q[i] = (unsigned) __float2int_rn( __fmul_rn( clamp1( x[i] ), 32767.0f ) ) & 0xFFFF;
		w[0] = q[0] | ( q[1] << 16 ); w[1] = q[2] | ( q[3] << 16 );
		}
	// pcm.c les2f_array: v * ( 1 / 0x8000 )
	static __device__ __forceinline__ void decode( const unsigned w[2], float x[4] )
		{
#pragma unroll
		for( int i = 0; i < 4; ++i ) x[i] = __fmul_rn( (float)(short)( w[i >> 1] >> ( 16 * ( i & 1 ) ) ), 1.0f / 32768.0f );
		}
	};

template<> struct Pcm<FLAN_B200_WAV_PCM_24>
	{
	static constexpr int BYTES = 3;
	// pcm.c f2let_array: lrintf( x * 0x7FFFFF ), low three bytes
	static __device__ __forceinline__ void encode( const float x[4], unsigned w[3] )
		{
		int q[4];
#pragma unroll
		for( int i = 0; i < 4; ++i ) q[i] = __float2int_rn( __fmul_rn( clamp1( x[i] ), 8388607.0f ) );
		pack4( q, w );
		}
	// pcm.c let2f_array: ( sample << 8 ) * ( 1 / 0x80000000 ) = sample / 2^23, exact in float
	static __device__ __forceinline__ void decode( const unsigned w[3], float x[4] )
		{
		int q[4];
		unpack4( w, q );
#pragma unroll
		for( int i = 0; i < 4; ++i ) x[i] = __fmul_rn( (float)( q[i] * 256 ), 1.0f / 2147483648.0f );
		}
	};

template<> struct Pcm<FLAN_B200_WAV_PCM_32>
	{
	static constexpr int BYTES = 4;
	// pcm.c f2lei_array: lrintf( x * 0x80000000 ). Full scale +1.0 gives 2^31, which x86 stores as INT_MIN (libsndfile's
	// int wraps; SSE cvtss2si returns its indefinite value); __float2int_rn would saturate to INT_MAX instead. NaN is
	// the SSE indefinite value INT_MIN too. Both are kept as the reference's platform gives them.
	static __device__ __forceinline__ void encode( const float x[4], unsigned w[4] )
		{
#pragma unroll
		for( int i = 0; i < 4; ++i )
			{
			const float s = clamp1( x[i] );
			w[i] = ( s == 1.0f || s != s ) ? 0x80000000u : (unsigned) __float2int_rn( __fmul_rn( s, 2147483648.0f ) );
			}
		}
	// pcm.c lei2f_array: v * ( 1 / 0x80000000 ); the int -> float conversion rounds to nearest even
	static __device__ __forceinline__ void decode( const unsigned w[4], float x[4] )
		{
#pragma unroll
		for( int i = 0; i < 4; ++i ) x[i] = __fmul_rn( __int2float_rn( (int) w[i] ), 1.0f / 2147483648.0f );
		}
	};

// A NaN keeps its payload on x86: the clamp's compares pass it through, and the float <-> double conversions keep the
// payload's top bits and set the quiet bit. Here the compiler may turn clamp1 into min / max, which return the canonical
// NaN, and the device conversions give the canonical NaN too; so the float types handle NaN on the bits.
__device__ __forceinline__ bool nan_bits( unsigned b ) { return ( b & 0x7FFFFFFFu ) > 0x7F800000u; }

template<> struct Pcm<FLAN_B200_WAV_FLOAT>
	{
	static constexpr int BYTES = 4;
	// float32.c: the bits of the (clamped) float, both ways
	static __device__ __forceinline__ void encode( const float x[4], unsigned w[4] )
		{
#pragma unroll
		for( int i = 0; i < 4; ++i )
			{
			const unsigned b = __float_as_uint( x[i] );
			w[i] = nan_bits( b ) ? b : __float_as_uint( clamp1( x[i] ) );
			}
		}
	static __device__ __forceinline__ void decode( const unsigned w[4], float x[4] )
		{
#pragma unroll
		for( int i = 0; i < 4; ++i ) x[i] = __uint_as_float( w[i] );
		}
	};

template<> struct Pcm<FLAN_B200_WAV_DOUBLE>
	{
	static constexpr int BYTES = 8;
	// double64.c: ( double ) x, exact; back: ( float ) d, round to nearest even (overflow to inf, gradual underflow).
	// NaN as x86's cvtss2sd / cvtsd2ss convert it: sign, quiet bit, the top 23 bits of the payload.
	static __device__ __forceinline__ void encode( const float x[4], unsigned w[8] )
		{
#pragma unroll
		for( int i = 0; i < 4; ++i )
			{
			const unsigned b = __float_as_uint( x[i] );
			const unsigned long long d = nan_bits( b )
				? ( (unsigned long long)( b & 0x80000000u ) << 32 ) | 0x7FF8000000000000ull | ( (unsigned long long)( b & 0x7FFFFFu ) << 29 )
				: (unsigned long long) __double_as_longlong( (double) clamp1( x[i] ) );
			w[2 * i] = (unsigned) d; w[2 * i + 1] = (unsigned)( d >> 32 );
			}
		}
	static __device__ __forceinline__ void decode( const unsigned w[8], float x[4] )
		{
#pragma unroll
		for( int i = 0; i < 4; ++i )
			{
			const unsigned long long d = ( (unsigned long long) w[2 * i + 1] << 32 ) | w[2 * i];
			x[i] = ( d & 0x7FFFFFFFFFFFFFFFull ) > 0x7FF0000000000000ull
				? __uint_as_float( ( w[2 * i + 1] & 0x80000000u ) | 0x7FC00000u | ( (unsigned)( d >> 29 ) & 0x7FFFFFu ) )
				: __double2float_rn( __longlong_as_double( (long long) d ) );
			}
		}
	};

// Interleaved value j = frame * C + channel <-> planar audio[channel * stride + frame]. A thread finds (frame, channel)
// of its first value once, then steps: by one value inside its four, by the grid's tile span from tile to tile.
struct Cursor
	{
	int64_t frame; int channel;
	__device__ Cursor( int64_t j, int C ) : frame( j / C ), channel( (int)( j % C ) ) {}
	__device__ __forceinline__ void next( int C ) { if( ++channel == C ) { channel = 0; ++frame; } }
	__device__ __forceinline__ void advance( const Cursor & by, int C )
		{
		frame += by.frame; channel += by.channel;
		if( channel >= C ) { channel -= C; ++frame; }
		}
	};

template<int T> __global__ void __launch_bounds__( THREADS ) pv_pcm_encode_kernel( const float * audio, int C, int64_t stride, int64_t n, uint8_t * bytes )
	{
	constexpr int W = Pcm<T>::BYTES;                    // words a thread = bytes a value
	__shared__ __align__( 16 ) unsigned tile[THREADS * W];
	const int64_t values = n * C;
	const int64_t tiles = ( values + TILE_VALUES - 1 ) / TILE_VALUES;
	Cursor at( (int64_t) blockIdx.x * TILE_VALUES + 4 * threadIdx.x, C );
	const Cursor span( (int64_t) gridDim.x * TILE_VALUES, C );
	for( int64_t t = blockIdx.x; t < tiles; t += gridDim.x, at.advance( span, C ) )
		{
		const int64_t v0 = t * TILE_VALUES + 4 * threadIdx.x;
		float x[4] = { 0.0f, 0.0f, 0.0f, 0.0f };
		Cursor c = at;
#pragma unroll
		for( int i = 0; i < 4; ++i )
			{
			if( v0 + i < values ) x[i] = __ldcs( audio + c.channel * stride + c.frame );
			c.next( C );
			}
		unsigned w[W];
		Pcm<T>::encode( x, w );
		put_words<W>( tile, w );
		__syncthreads();
		store_tile<W>( tile, bytes, t, values * W );
		__syncthreads();
		}
	}

template<int T> __global__ void __launch_bounds__( THREADS ) pv_pcm_decode_kernel( const uint8_t * bytes, int C, int64_t stride, int64_t n, float * audio )
	{
	constexpr int W = Pcm<T>::BYTES;
	__shared__ __align__( 16 ) unsigned tile[THREADS * W];
	const int64_t values = n * C;
	const int64_t tiles = ( values + TILE_VALUES - 1 ) / TILE_VALUES;
	Cursor at( (int64_t) blockIdx.x * TILE_VALUES + 4 * threadIdx.x, C );
	const Cursor span( (int64_t) gridDim.x * TILE_VALUES, C );
	for( int64_t t = blockIdx.x; t < tiles; t += gridDim.x, at.advance( span, C ) )
		{
		load_tile<W>( tile, bytes, t, values * W );
		__syncthreads();
		unsigned w[W];
		get_words<W>( tile, w );
		float x[4];
		Pcm<T>::decode( w, x );
		const int64_t v0 = t * TILE_VALUES + 4 * threadIdx.x;
		Cursor c = at;
#pragma unroll
		for( int i = 0; i < 4; ++i )
			{
			if( v0 + i < values ) audio[c.channel * stride + c.frame] = x[i];
			c.next( C );
			}
		__syncthreads();
		}
	}

static unsigned grid_for( int64_t values, int sms )
	{
	int64_t tiles = ( values + TILE_VALUES - 1 ) / TILE_VALUES;
	if( tiles > (int64_t) sms * 16 ) tiles = (int64_t) sms * 16;
	return (unsigned)( tiles < 1 ? 1 : tiles );
	}

cudaError_t launch_flan_encode( const float * pv, int64_t count, float dft_size, float sample_rate, uint8_t * bytes, int sms, cudaStream_t st )
	{
	pv_flan_encode_kernel<<<grid_for( 2 * count, sms ), THREADS, 0, st>>>( pv, 2 * count, dft_size, sample_rate, bytes );
	return cudaGetLastError();
	}
cudaError_t launch_flan_decode( const uint8_t * bytes, int64_t count, float dft_size, float sample_rate, float * pv, int sms, cudaStream_t st )
	{
	pv_flan_decode_kernel<<<grid_for( 2 * count, sms ), THREADS, 0, st>>>( bytes, 2 * count, dft_size, sample_rate, pv );
	return cudaGetLastError();
	}

int pcm_width( int subtype )
	{
	switch( subtype )
		{
		case FLAN_B200_WAV_PCM_U8: return Pcm<FLAN_B200_WAV_PCM_U8>::BYTES;
		case FLAN_B200_WAV_PCM_16: return Pcm<FLAN_B200_WAV_PCM_16>::BYTES;
		case FLAN_B200_WAV_PCM_24: return Pcm<FLAN_B200_WAV_PCM_24>::BYTES;
		case FLAN_B200_WAV_PCM_32: return Pcm<FLAN_B200_WAV_PCM_32>::BYTES;
		case FLAN_B200_WAV_FLOAT: return Pcm<FLAN_B200_WAV_FLOAT>::BYTES;
		case FLAN_B200_WAV_DOUBLE: return Pcm<FLAN_B200_WAV_DOUBLE>::BYTES;
		default: return 0;
		}
	}

#define PVIO_EACH_SUBTYPE( X ) X( FLAN_B200_WAV_PCM_U8 ) X( FLAN_B200_WAV_PCM_16 ) X( FLAN_B200_WAV_PCM_24 ) \
                               X( FLAN_B200_WAV_PCM_32 ) X( FLAN_B200_WAV_FLOAT ) X( FLAN_B200_WAV_DOUBLE )

cudaError_t launch_pcm_encode( int subtype, const float * audio, int C, int64_t stride, int64_t n, uint8_t * bytes, int sms, cudaStream_t st )
	{
	const unsigned grid = grid_for( n * C, sms );
	switch( subtype )
		{
#define PVIO_CASE( T ) case T: pv_pcm_encode_kernel<T><<<grid, THREADS, 0, st>>>( audio, C, stride, n, bytes ); break;
		PVIO_EACH_SUBTYPE( PVIO_CASE )
#undef PVIO_CASE
		default: return cudaErrorInvalidValue;
		}
	return cudaGetLastError();
	}

cudaError_t launch_pcm_decode( int subtype, const uint8_t * bytes, int C, int64_t stride, int64_t n, float * audio, int sms, cudaStream_t st )
	{
	const unsigned grid = grid_for( n * C, sms );
	switch( subtype )
		{
#define PVIO_CASE( T ) case T: pv_pcm_decode_kernel<T><<<grid, THREADS, 0, st>>>( bytes, C, stride, n, audio ); break;
		PVIO_EACH_SUBTYPE( PVIO_CASE )
#undef PVIO_CASE
		default: return cudaErrorInvalidValue;
		}
	return cudaGetLastError();
	}

} // namespace pvio
