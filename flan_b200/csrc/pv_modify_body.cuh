// flan_b200/csrc/pv_modify_body.cuh
//
// Bodies of the PV-domain kernels that sit between analysis and resynthesis (BASELINE config 4): PV::repitch /
// PV::modify_frequency (reference PV/PVModify.cpp:196-305) and PV::stretch / PV::modify_time (PVModify.cpp:307-385).
// Integer / float work whose results must be bit-identical to the reference: every float expression below keeps the
// reference's operation order and this file is compiled without FMA contraction (nvcc -fmad=false, g++
// -ffp-contract=off), with IEEE division and square root. Written as per-thread phase functions between barriers so
// that the identical source runs on the device (pv_modify.cu) and, thread by thread, in the CPU emulator
// (emu/pv_emu.cpp) used by the tests in a container without a GPU.
//
// Frame x bin tables (the reference's FunctionSample2d, PV/PV.h:31-35) are passed as strided views: element
// (frame, bin) = p[frame * frame_stride + bin * bin_stride]. (B,1) is a full table, (0,1) one row shared by all
// frames, (1,0) one column shared by all bins, (0,0) a single value.
//
// Both reference algorithms walk sequentially and scatter: repitch walks the bin pairs of a frame in order and writes
// output bins with an order-dependent rule (PVModify.cpp:237-243); stretch walks the frame pairs of a bin in order
// and accumulates into output frames (PVModify.cpp:353-355). When the mapped positions are monotone along the walk,
// consecutive pairs write DISJOINT output ranges ([ceil(lo), ceil(hi)) abut), every output cell is written at most
// once, starting from zero, and the walk order no longer matters: those rows / columns run fully parallel and
// bit-exact. Anything else takes the sequential walk.
#pragma once

#include <cstdint>
#include <cmath>

#include "pv_core.cuh"      // PhaseSegAcc: the phase summary a producing kernel leaves behind for PV::convert_to_audio

#if defined( __CUDACC__ )
#include <cuda_runtime.h>
#define PVM_HD __host__ __device__ __forceinline__
#else
#include <vector_types.h>
#include <vector_functions.h>
#define PVM_HD inline
#endif

namespace pvm {

struct Table
	{
	const float * p;
	int64_t frame_stride;
	int bin_stride;
	PVM_HD float at( int64_t frame, int bin ) const { return p[frame * frame_stride + (int64_t) bin * bin_stride]; }
	};

// Utility/Interpolator.cpp:15-101. ids: 0 linear, 1 midpoint, 2 nearest, 3 floor, 4 ceil, 5 smoothstep,
// 6 smootherstep, 7 sine, 8 sine2, 9 sqrt. 7 is cosf in the reference (evaluated here in double and rounded: the
// correctly rounded value, which glibc's cosf returns for all but a few inputs per thousand); 8 is double sin there too.
PVM_HD float interp_eval( int id, float x )
	{
	const float pi = 3.14159274101257324f;      // acosf( -1.0f ), Interpolator.cpp:8
	const float sqrt2 = 1.41421353816986084f;   // sqrtf( 2.0f ), Interpolator.cpp:9
	switch( id )
		{
		case 1: return 0.5f;
		case 2: return roundf( x );
		case 3: return 0.0f;
		case 4: return 1.0f;
		case 5: return x * x * ( 3.0f - 2.0f * x );
		case 6: return x * x * x * ( x * ( x * 6.0f - 15.0f ) + 10.0f );
		case 7: return ( 1.0f - (float) cos( (double)( pi * x ) ) ) / 2.0f;
		case 8: return (float)( (double) sqrt2 * sin( (double)( pi / 4.0f * x ) ) );
		case 9: return sqrtf( x );
		default: return x;
		}
	}

PVM_HD int clampi( int v, int lo, int hi ) { return v < lo ? lo : ( hi < v ? hi : v ); }
// float -> int the way the reference's x86 build converts in range; out-of-range / NaN inputs (undefined there) saturate.
PVM_HD int to_int( float v )
	{
	if( !( v > -2147483648.0f ) ) return INT32_MIN;
	if( !( v < 2147483648.0f ) ) return INT32_MAX;
	return (int) v;
	}

// ------------------------------------------------------------------------------------------------
// repitch / modify_frequency: one CTA per (channel, frame) row.
// ------------------------------------------------------------------------------------------------
struct RepitchArgs
	{
	const float2 * pv;          // [C][F][B]
	float2 * out;               // [C][F][B]
	Table mod;                  // mapped bin positions in Hz (PVModify.cpp:217-219), shared by all channels
	const float * in_mod;       // [C][F][B] mapped frequency of every input MF (modify_frequency), or null: the lerp of
	                            // PV::repitch (PVModify.cpp:289-302) is evaluated from `mod`
	int64_t F;
	int B;
	float bin_width;            // sample_rate / float( dft ), PVBuffer.cpp:438-441
	int interp;
	};

// Shared-memory view of one row: five float arrays of B elements, then the output row.
struct RepitchRow
	{
	float * hz; float * pos; float * m; float * fm; float2 * out;
	PVM_HD static size_t bytes( int B ) { return sizeof( float ) * 4 * (size_t)( B + 1 ) + sizeof( float2 ) * (size_t) B + 8; }
	PVM_HD RepitchRow( void * base, int B )
		{
		out = (float2 *) base;
		hz = (float *)( out + B ); pos = hz + B + 1; m = pos + B + 1; fm = m + B + 1;
		}
	};

// Phase 1: stage the row. fm holds the raw input frequency until phase 2.
PVM_HD void repitch_load( const RepitchArgs & a, int64_t row, int tid, int nt, RepitchRow & s )
	{
	const int64_t frame = row % a.F;
	const float2 * in = a.pv + row * a.B;
	for( int b = tid; b < a.B; b += nt )
		{
		const float hz = a.mod.at( frame, b );
		const float2 mf = in[b];
		s.hz[b] = hz;
		s.pos[b] = hz / a.bin_width;                                    // frequency_to_bin, PVModify.cpp:218-219
		s.m[b] = mf.x;
		s.fm[b] = a.in_mod ? a.in_mod[row * a.B + b] : mf.y;
		s.out[b] = make_float2( 0.0f, 0.0f );                           // out.clear_buffer(), PVModify.cpp:205
		}
	}

// Phase 2: PV::repitch's lerp of the integrated factor at each MF's own frequency (PVModify.cpp:293-299), plus this
// thread's share of the monotonicity test. Returns bit 0: some pair descends (or is NaN), bit 1: some pair ascends (or NaN).
PVM_HD int repitch_map( const RepitchArgs & a, int tid, int nt, RepitchRow & s )
	{
	int flags = 0;
	const float top = (float)( a.B - 1 ) - 0.0001f;
	for( int b = tid; b < a.B; b += nt )
		{
		if( !a.in_mod )
			{
			float fbin = s.fm[b] / a.bin_width;
			fbin = fbin < 0.0f ? 0.0f : ( top < fbin ? top : fbin );    // std::clamp
			const int lo = clampi( to_int( floorf( fbin ) ), 0, a.B - 2 );   // the clamp only matters for NaN input
			const float lo_freq = s.hz[lo], hi_freq = s.hz[lo + 1];
			const float r = fbin - (float) lo;
			s.fm[b] = lo_freq * ( 1.0f - r ) + hi_freq * r;
			}
		if( b > 0 )
			{
			const float lo = s.pos[b - 1], hi = s.pos[b];
			if( !( hi >= lo ) ) flags |= 1;
			if( !( hi <= lo ) ) flags |= 2;
			}
		}
	return flags;
	}
// fm[b] is rewritten in place while other threads read hz only, so phases 1 and 2 need one barrier between them and
// phase 3 one after the vote.

// One adjacent bin pair (PVModify.cpp:214-244).
PVM_HD void repitch_pair( const RepitchArgs & a, int bin, RepitchRow & s )
	{
	const float loBin = s.pos[bin - 1], hiBin = s.pos[bin];
	const bool forward = hiBin > loBin;
	const int start = clampi( to_int( forward ? ceilf( loBin ) : floorf( loBin ) ), 0, a.B - 1 );
	const int end = clampi( to_int( forward ? ceilf( hiBin ) : floorf( hiBin ) ), 0, a.B - 1 );
	if( forward ? start >= end : start <= end ) return;
	const float lo_m = s.m[bin - 1], lo_f = s.fm[bin - 1], hi_m = s.m[bin], hi_f = s.fm[bin];
	const float den = hiBin - loBin;
	const int step = forward ? 1 : -1;
	for( int y = start; y != end; y += step )
		{
		const float mix = interp_eval( a.interp, ( (float) y - loBin ) / den );
		const float w0 = ( 1.0f - mix ) * lo_m;
		const float w1 = mix * hi_m;
		const bool lo_wins = w0 < w1;
		const float mm = lo_wins ? lo_m : hi_m, ff = lo_wins ? lo_f : hi_f;
		float2 o = s.out[y];
		if( mm > o.x )
			{
			o.x = o.x + mm;
			o.y = ff;
			s.out[y] = o;
			}
		}
	}

// Phase 3. flags = OR over the CTA of repitch_map's result.
PVM_HD void repitch_scatter( const RepitchArgs & a, int flags, int tid, int nt, RepitchRow & s )
	{
	if( flags != 3 )
		for( int bin = 1 + tid; bin < a.B; bin += nt ) repitch_pair( a, bin, s );      // disjoint ranges
	else if( tid == 0 )
		for( int bin = 1; bin < a.B; ++bin ) repitch_pair( a, bin, s );                // the reference's walk
	}

// Phase 4.
PVM_HD void repitch_store( const RepitchArgs & a, int64_t row, int tid, int nt, RepitchRow & s )
	{
	float2 * out = a.out + row * a.B;
	for( int b = tid; b < a.B; b += nt ) out[b] = s.out[b];
	}

// ------------------------------------------------------------------------------------------------
// repitch, frame-shared table (a constant or frequency-only factor): the mapped positions, hence every pair's output
// range and every output bin's mix value, are the same for all rows. A one-CTA plan kernel evaluates them once; when
// the positions are monotone each output bin has at most ONE source pair and the row kernel becomes a gather:
//     out[y] = select( (1-mix[y]) * m[p-1] < mix[y] * m[p] ) ...   with p = src[y]
// which is exactly what the reference's walk leaves in a zero-initialised row (PVModify.cpp:232-243 with outMF = 0).
// ------------------------------------------------------------------------------------------------
struct RepitchPlan
	{
	int * src;                  // [B] upper bin of the pair that covers output bin y; 0 = none
	float * mix;                // [B] interp( ( y - loBin ) / ( hiBin - loBin ) ) of that pair
	int * ok;                   // 1: plan valid (monotone positions); 0: rows must take the general kernel
	};

// Plan phases (one CTA; `pos` is a B-float scratch in shared memory).
PVM_HD int repitch_plan_positions( const float * hz, int B, float bin_width, int tid, int nt, float * pos, const RepitchPlan & plan )
	{
	for( int b = tid; b < B; b += nt ) { pos[b] = hz[b] / bin_width; plan.src[b] = 0; plan.mix[b] = 0.0f; }
	return 0;
	}
PVM_HD int repitch_plan_flags( int B, int tid, int nt, const float * pos )
	{
	int flags = 0;
	for( int b = 1 + tid; b < B; b += nt )
		{
		const float lo = pos[b - 1], hi = pos[b];
		if( !( hi >= lo ) ) flags |= 1;
		if( !( hi <= lo ) ) flags |= 2;
		}
	return flags;
	}
PVM_HD void repitch_plan_pairs( int B, int interp, int flags, int tid, int nt, const float * pos, const RepitchPlan & plan )
	{
	if( tid == 0 ) *plan.ok = flags != 3;
	if( flags == 3 ) return;
	for( int bin = 1 + tid; bin < B; bin += nt )
		{
		const float loBin = pos[bin - 1], hiBin = pos[bin];
		const bool forward = hiBin > loBin;
		const int start = clampi( to_int( forward ? ceilf( loBin ) : floorf( loBin ) ), 0, B - 1 );
		const int end = clampi( to_int( forward ? ceilf( hiBin ) : floorf( hiBin ) ), 0, B - 1 );
		if( forward ? start >= end : start <= end ) continue;
		const float den = hiBin - loBin;
		const int step = forward ? 1 : -1;
		for( int y = start; y != end; y += step )
			{
			plan.src[y] = bin;
			plan.mix[y] = interp_eval( interp, ( (float) y - loBin ) / den );
			}
		}
	}

// Row phases of the gather kernel. m / fm: shared-memory rows of B floats (double-buffered by the caller).
PVM_HD float repitch_lerp( const float * hz, int B, float bin_width, float f )
	{
	const float top = (float)( B - 1 ) - 0.0001f;
	float fbin = f / bin_width;
	fbin = fbin < 0.0f ? 0.0f : ( top < fbin ? top : fbin );
	const int lo = clampi( to_int( floorf( fbin ) ), 0, B - 2 );
	const float r = fbin - (float) lo;
	return hz[lo] * ( 1.0f - r ) + hz[lo + 1] * r;
	}
PVM_HD float2 repitch_gather( int y, const int * src, const float * mix, const float * m, const float * fm )
	{
	const int p = src[y];
	if( p == 0 ) return make_float2( 0.0f, 0.0f );
	const float mx = mix[y];
	const float lo_m = m[p - 1], hi_m = m[p];
	const float w0 = ( 1.0f - mx ) * lo_m;
	const float w1 = mx * hi_m;
	const bool lo_wins = w0 < w1;
	const float mm = lo_wins ? lo_m : hi_m;
	if( !( mm > 0.0f ) ) return make_float2( 0.0f, 0.0f );
	return make_float2( 0.0f + mm, lo_wins ? fm[p - 1] : fm[p] );
	}

// ------------------------------------------------------------------------------------------------
// Table preparation
// ------------------------------------------------------------------------------------------------
// PV::repitch: running sum of the factor along bins, then bin_to_frequency (PVModify.cpp:278-284). One thread per row.
PVM_HD void bin_prefix_row( const Table & factor, int64_t row, int B, float sample_rate, float dft, float * out_row )
	{
	float acc = 0.0f;
	for( int b = 0; b < B; ++b )
		{
		const float v = factor.at( row, b );
		acc = b == 0 ? v : v + acc;
		out_row[b] = acc * sample_rate / dft;                           // PVBuffer.cpp:443-446
		}
	}

// Order-preserving unsigned key of a float, for atomicMax.
PVM_HD uint32_t float_key( float f )
	{
	uint32_t u;
#if defined( __CUDA_ARCH__ )
	u = __float_as_uint( f );
#else
	union { float f; uint32_t u; } c; c.f = f; u = c.u;
#endif
	return ( u & 0x80000000u ) ? ~u : ( u | 0x80000000u );
	}
PVM_HD float key_float( uint32_t k )
	{
	const uint32_t u = ( k & 0x80000000u ) ? ( k & 0x7fffffffu ) : ~k;
#if defined( __CUDA_ARCH__ )
	return __uint_as_float( u );
#else
	union { float f; uint32_t u; } c; c.u = u; return c.f;
#endif
	}

// PV::stretch: running sum of the factor along frames (PVModify.cpp:376-378) -- the one inherently sequential step
// (float addition does not re-associate): one thread per column, nothing but the add and a store in its loop.
PVM_HD void frame_prefix_column( const Table & factor, int col, int64_t F, int cols, float * out )
	{
	const float * src = factor.p + (int64_t) col * factor.bin_stride;
	float * dst = out + col;
	float acc = 0.0f;
	constexpr int U = 16;       // the loads of a batch are issued together, ahead of the dependent chain of adds
	int64_t f = 0;
	for( ; f + U <= F; f += U )
		{
		float v[U];
#pragma unroll
		for( int j = 0; j < U; ++j ) v[j] = src[j * factor.frame_stride];
#pragma unroll
		for( int j = 0; j < U; ++j ) { acc = ( f + j == 0 ) ? v[j] : v[j] + acc; v[j] = acc; }
#pragma unroll
		for( int j = 0; j < U; ++j ) dst[(int64_t) j * cols] = v[j];
		src += U * factor.frame_stride; dst += (int64_t) U * cols;
		}
	for( ; f < F; ++f, src += factor.frame_stride, dst += cols )
		{
		acc = f == 0 ? *src : *src + acc;
		*dst = acc;
		}
	}

// Constant factor: acc[k] = fl( acc[k-1] + c ) has a closed form per binade. Inside [2^e, 2^(e+1)) every value is a
// multiple of u = ulp, so fl( x + c ) = x + u * round( c / u ) with the SAME increment for every x -- except that an
// exact tie ( c / u = n + 1/2 ) rounds to even and the first step in the binade may differ by one ulp, after which the
// parity, hence the increment, is fixed. So: take real float steps until two consecutive increments inside one binade
// agree, then jump to the end of the binade in one go. A few steps per binade instead of F dependent additions; the
// values are then filled in parallel from the segment list, bit-identical to the sequential sum.
struct PrefixSeg { int64_t k0; int64_t n; double a0; double d; };      // acc[k0 + i] = float( a0 + i * d ), 0 <= i < n
constexpr int PREFIX_MAX_SEGS = 1024;

PVM_HD uint32_t float_bits( float f )
	{
#if defined( __CUDA_ARCH__ )
	return __float_as_uint( f );
#else
	union { float f; uint32_t u; } c; c.f = f; return c.u;
#endif
	}
PVM_HD int exponent_field( float x ) { return (int)( ( float_bits( x ) >> 23 ) & 0xffu ); }

// Single thread. Segments describe |acc|; the fill applies the sign of c. Returns the segment count.
PVM_HD int constant_prefix_segments( float c, int64_t F, PrefixSeg * segs )
	{
	const float a = fabsf( c );
	int ns = 0;
	auto emit = [&]( int64_t k0, int64_t n, double a0, double d ) { if( ns < PREFIX_MAX_SEGS ) segs[ns] = PrefixSeg{ k0, n, a0, d }; ++ns; };
	if( F < 1 ) return 0;
	emit( 0, 1, a, 0.0 );
	int64_t k = 0;                  // last index produced
	float x0 = a;                   // its value
	while( k < F - 1 )
		{
		if( !( x0 < INFINITY ) || ns >= PREFIX_MAX_SEGS - 2 )      // inf / NaN are absorbing; segment budget: finish sequentially in spirit
			{
			if( !( x0 < INFINITY ) ) { emit( k + 1, F - 1 - k, x0 + a, 0.0 ); return ns; }
			}
		const float x1 = x0 + a, x2 = x1 + a;
		const int e = exponent_field( x0 );
		const double d01 = (double) x1 - (double) x0, d12 = (double) x2 - (double) x1;
		if( e != 0xff && exponent_field( x1 ) == e && exponent_field( x2 ) == e && d01 == d12 )
			{
			int64_t cnt;                                           // values x1, x1 + d, ... produced by this run
			if( d12 == 0.0 ) cnt = F - 1 - k;
			else
				{
				const double u = ldexp( 1.0, ( e ? e : 1 ) - 150 );    // ulp of the binade (denormals share 2^-149)
				const double top = ldexp( 1.0, ( e ? e : 1 ) - 126 );
				const int64_t steps = (int64_t) floor( ( top - u - (double) x1 ) / d12 );     // valid steps from x1
				cnt = steps + 1;
				if( cnt > F - 1 - k ) cnt = F - 1 - k;
				}
			emit( k + 1, cnt, (double) x1, d12 );
			k += cnt;
			x0 = (float)( (double) x1 + (double)( cnt - 1 ) * d12 );
			}
		else
			{
			emit( k + 1, 1, (double) x1, 0.0 );
			k += 1;
			x0 = x1;
			}
		}
	return ns;
	}

// Value at index k from the segment list (binary search), with the sign of c.
PVM_HD float constant_prefix_value( const PrefixSeg * segs, int ns, float c, int64_t k )
	{
	int lo = 0, hi = ns - 1;
	while( lo < hi )
		{
		const int mid = ( lo + hi + 1 ) >> 1;
		if( segs[mid].k0 <= k ) lo = mid; else hi = mid - 1;
		}
	const float v = (float)( segs[lo].a0 + (double)( k - segs[lo].k0 ) * segs[lo].d );
	return c < 0.0f ? -v : v;
	}

// ... then frame_to_time (PVModify.cpp:381-382, PVBuffer.cpp:433-436) element-wise, raw sums -> seconds.
PVM_HD void frame_prefix_convert( const float * raw, float * out, int64_t i, float rate )
	{
	out[i] = raw[i] / rate;
	}

// ------------------------------------------------------------------------------------------------
// stretch / modify_time
// ------------------------------------------------------------------------------------------------
struct StretchArgs
	{
	const float2 * pv;          // [C][F][B]
	float2 * out;               // [C][out_frames][B]
	Table mod;                  // seconds (PVModify.cpp:331-332)
	int64_t F, out_frames;
	int B;
	float sample_rate, hop;     // time_to_frame( t ) = t * sample_rate / float( hop ), PVBuffer.cpp:428-431
	int interp;
	int chunk;                  // frame pairs per thread in the parallel form
	int64_t chunks;
	// Planned form only: a window of the rows, so that one launch writes the segments of one output shard (pv_capi_multi.cu).
	// pv holds input frames [row0, ...) with pv_channel_stride MF between channels, out holds output frames
	// [out_row0, ...) with out_channel_stride; the launch's segments are seg0, seg0 + 1, ... Whole signal: 0, F * B, 0,
	// out_frames * B, 0.
	int64_t row0, pv_channel_stride;
	int64_t out_row0, out_channel_stride;
	int64_t seg0;
	};

PVM_HD float time_to_frame( const StretchArgs & a, float t ) { return t * a.sample_rate / a.hop; }

// One adjacent frame pair of one (channel, bin) column (PVModify.cpp:329-357). RMW = the reference's accumulate into
// whatever earlier pairs left in the output; !RMW = the output cells are known to be untouched (zero): the same
// expressions evaluated on zeros, and every covered cell is written, zeros included.
template<bool RMW>
PVM_HD void stretch_pair( const StretchArgs & a, float2 * out_col, float lFrame, float rFrame, float2 l, float2 r )
	{
	const bool forward = rFrame > lFrame;
	int start = to_int( forward ? ceilf( lFrame ) : floorf( lFrame ) );
	int end = to_int( forward ? ceilf( rFrame ) : floorf( rFrame ) );
	const int64_t last = a.out_frames - 1;
	// frames outside [0, out_frames) are skipped before anything is computed (PVModify.cpp:343)
	if( forward )
		{
		if( start < 0 ) start = 0;
		if( (int64_t) end > a.out_frames ) end = (int) a.out_frames;
		if( start >= end ) return;
		}
	else
		{
		if( (int64_t) start > last ) start = (int) last;
		if( end < -1 ) end = -1;
		if( start <= end ) return;
		}
	const float den = rFrame - lFrame;
	const int step = forward ? 1 : -1;
	bool live = true;
	for( int x = start; x != end; x += step )
		{
		float2 * o = out_col + (int64_t) x * a.B;
		if( live )
			{
			const float mix = interp_eval( a.interp, ( (float) x - lFrame ) / den );
			const float w0 = ( 1.0f - mix ) * l.x;
			const float w1 = mix * r.x;
			const float totalWeight = w0 + w1;
			const float weightedFreqSum = w0 * l.y + w1 * r.y;
			if( totalWeight == 0.0f ) live = false;                     // `return`: leaves this frame pair (PVModify.cpp:351-352)
			else
				{
				const float2 old = RMW ? *o : make_float2( 0.0f, 0.0f );
				float2 nw;
				nw.y = ( old.y * old.x + weightedFreqSum ) / ( old.x + totalWeight );
				nw.x = old.x + totalWeight;
				*o = nw;
				continue;
				}
			}
		if( RMW ) return;
		*o = make_float2( 0.0f, 0.0f );
		}
	}

// Parallel form (every column non-descending): thread = (channel, chunk of frame pairs, bin). Covered output frames
// are written by their pair; the first / last chunk also clear what lies below / above the column's covered range.
PVM_HD void stretch_chunk( const StretchArgs & a, int c, int64_t chunk_index, int bin )
	{
	const float2 * in = a.pv + (int64_t) c * a.F * a.B + bin;
	float2 * out_col = a.out + (int64_t) c * a.out_frames * a.B + bin;
	const int64_t f0 = chunk_index * a.chunk;                           // pairs (f0, f0+1) ... (f1-1, f1)
	int64_t f1 = f0 + a.chunk;
	if( f1 > a.F - 1 ) f1 = a.F - 1;
	float lF = time_to_frame( a, a.mod.at( f0, bin ) );
	float2 l = in[f0 * a.B];
	if( chunk_index == 0 )
		{
		int64_t head = to_int( ceilf( lF ) );
		if( head > a.out_frames ) head = a.out_frames;
		for( int64_t x = 0; x < head; ++x ) out_col[x * a.B] = make_float2( 0.0f, 0.0f );
		}
	constexpr int BATCH = 8;
	for( int64_t f = f0; f < f1; f += BATCH )
		{
		float2 r[BATCH]; float rF[BATCH];
#pragma unroll
		for( int j = 0; j < BATCH; ++j )
			if( f + 1 + j <= f1 )
				{
				r[j] = in[( f + 1 + j ) * a.B];
				rF[j] = time_to_frame( a, a.mod.at( f + 1 + j, bin ) );
				}
#pragma unroll
		for( int j = 0; j < BATCH; ++j )
			if( f + 1 + j <= f1 )
				{
				stretch_pair<false>( a, out_col, lF, rF[j], l, r[j] );
				l = r[j]; lF = rF[j];
				}
		}
	if( chunk_index == a.chunks - 1 )
		{
		int64_t tail = to_int( ceilf( lF ) );                           // lF is now the position of frame F-1
		if( tail < 0 ) tail = 0;
		for( int64_t x = tail; x < a.out_frames; ++x ) out_col[x * a.B] = make_float2( 0.0f, 0.0f );
		}
	}

// Bin-shared time map (a constant or time-only factor), never descending: the pair geometry is the same for every
// bin, so it is evaluated once by a plan kernel -- xpos[f] = first output frame at or after frame f's mapped position,
// clamped to [0, out_frames]; pair (f-1, f) covers [xpos[f-1], xpos[f]) -- together with mix[x] of every covered
// output frame. The chunk kernel then only does the per-bin arithmetic of PVModify.cpp:346-355.
struct StretchPlan
	{
	int * xpos;                 // [F]
	float * mix;                // [out_frames]
	int * src;                  // [out_frames] the frame f whose pair (f-1, f) covers the output frame; -1 (preset) where none does
	};

PVM_HD void stretch_plan_frame( const StretchArgs & a, const StretchPlan & plan, int64_t f )
	{
	const float pos = time_to_frame( a, a.mod.at( f, 0 ) );
	int64_t x = to_int( ceilf( pos ) );
	x = x < 0 ? 0 : ( x > a.out_frames ? a.out_frames : x );
	plan.xpos[f] = (int) x;
	if( f == 0 ) return;
	const float lFrame = time_to_frame( a, a.mod.at( f - 1, 0 ) );
	if( !( pos > lFrame ) ) return;
	int64_t xs = to_int( ceilf( lFrame ) );
	xs = xs < 0 ? 0 : xs;
	const float den = pos - lFrame;
	for( ; xs < x; ++xs ) { plan.mix[xs] = interp_eval( a.interp, ( (float) xs - lFrame ) / den ); plan.src[xs] = (int) f; }
	}

// Input rows [*r0, *r1) that stretch_segment_planned reads for the output frames [x0, x1): the frames of the pairs that
// cover them, and the left frame of the first -- the pair a segment that begins inside it looks back into. Empty when no
// pair covers any of them (zeros below xpos[0] and above xpos[F-1]).
PVM_HD void stretch_window( const StretchPlan & plan, int64_t F, int64_t x0, int64_t x1, int64_t * r0, int64_t * r1 )
	{
	int64_t c0 = plan.xpos[0], c1 = plan.xpos[F - 1];
	if( c0 < x0 ) c0 = x0;
	if( c1 > x1 ) c1 = x1;
	if( c0 >= c1 ) { *r0 = 0; *r1 = 0; return; }
	*r0 = plan.src[c0] - 1;
	*r1 = plan.src[c1 - 1] + 1;
	}

// The same arithmetic by OUTPUT segments: thread = (channel, run of seg_len output frames, bin) gathers its frames in
// increasing order -- the order in which PV::convert_to_audio accumulates the phase of a bin (phase_vocoder.cpp:57-59)
// -- so it can leave the segment's phase summary behind (summary != null) and resynthesis need not read the rows again.
// A segment that begins inside a pair first re-evaluates whether an earlier frame of the pair ended it
// (`return` at PVModify.cpp:351-352).
template<bool SUMM>
PVM_HD void stretch_segment_planned( const StretchArgs & a, const StretchPlan & plan, int c, int64_t seg, int seg_len, int bin,
                                     pvk::PhaseSegAcc * summary, const pvk::PvConsts & k )
	{
	const float2 * in = a.pv + (int64_t) c * a.pv_channel_stride + bin;
	const int64_t B = a.B;
	int x = (int)( ( a.seg0 + seg ) * seg_len );                        // the planned form runs below 2^31 frames
	int x1 = x + seg_len;
	if( (int64_t) x1 > a.out_frames ) x1 = (int) a.out_frames;
	float2 * o = a.out + (int64_t) c * a.out_channel_stride + ( x - a.out_row0 ) * B + bin;     // the output cell of frame x
	const float2 zero = make_float2( 0.0f, 0.0f );
	// The pairs cover [xpos[0], xpos[F-1]) without gaps (the map never descends): zeros below, pairs f_lo .. f_hi, zeros above.
	int c0 = plan.xpos[0], c1 = plan.xpos[a.F - 1];
	if( c0 > x1 ) c0 = x1;
	if( c1 > x1 ) c1 = x1;
	if( c1 < x ) c1 = x;
	for( ; x < c0; ++x, o += B ) *o = zero;                              // a zero row adds nothing to the phase summary
	if( x < c1 )
		{
		const int f_lo = plan.src[x], f_hi = plan.src[c1 - 1];
		const float2 * row = in + ( f_lo - a.row0 ) * B;                // right frame of the current pair
		float2 l = *( row - B );
		bool live = true;
		// a segment that begins inside a pair: did an earlier frame of the pair end it (PVModify.cpp:351-352)?
		const int z0 = plan.xpos[f_lo - 1];
		if( z0 < x )
			{
			const float2 r = *row;
			for( int z = z0; z < x && live; ++z )
				{
				const float mix = plan.mix[z];
				const float w0 = ( 1.0f - mix ) * l.x;
				const float w1 = mix * r.x;
				if( w0 + w1 == 0.0f ) live = false;
				}
			}
		constexpr int BATCH = SUMM ? 4 : 8;
		const int * xp = plan.xpos + f_lo;
		const float * mixp = plan.mix + x;
		for( int f = f_lo; f <= f_hi; f += BATCH, xp += BATCH )
			{
			float2 r[BATCH]; int xe[BATCH];
#pragma unroll
			for( int j = 0; j < BATCH; ++j )
				if( f + j <= f_hi )
					{
					r[j] = row[(int64_t) j * B];
					xe[j] = xp[j];
					}
			row += (int64_t) BATCH * B;
#pragma unroll
			for( int j = 0; j < BATCH; ++j )
				if( f + j <= f_hi )
					{
					const int xend = xe[j] < c1 ? xe[j] : c1;
					if( live )
						for( ; x < xend; ++x, o += B, ++mixp )
							{
							const float mix = *mixp;
							const float w0 = ( 1.0f - mix ) * l.x;
							const float w1 = mix * r[j].x;
							const float totalWeight = w0 + w1;
							const float weightedFreqSum = w0 * l.y + w1 * r[j].y;
							if( totalWeight == 0.0f ) break;                        // leaves this frame pair (PVModify.cpp:351-352)
							float2 nw;
							nw.y = ( 0.0f * 0.0f + weightedFreqSum ) / ( 0.0f + totalWeight );
							nw.x = 0.0f + totalWeight;
							*o = nw;
							if( SUMM ) summary->step<true>( nw, k );
							}
					// what is left of a pair that ended early stays zero (a zero row adds nothing to the phase summary)
					for( ; x < xend; ++x, o += B, ++mixp ) *o = zero;
					l = r[j];
					live = true;
					}
			}
		}
	for( ; x < x1; ++x, o += B ) *o = zero;
	}

// Sequential form (the reference's walk): thread = (channel, bin); the output was cleared beforehand.
PVM_HD void stretch_column( const StretchArgs & a, int c, int bin )
	{
	const float2 * in = a.pv + (int64_t) c * a.F * a.B + bin;
	float2 * out_col = a.out + (int64_t) c * a.out_frames * a.B + bin;
	float lF = time_to_frame( a, a.mod.at( 0, bin ) );
	float2 l = in[0];
	for( int64_t f = 1; f < a.F; ++f )
		{
		const float rF = time_to_frame( a, a.mod.at( f, bin ) );
		const float2 r = in[f * a.B];
		stretch_pair<true>( a, out_col, lF, rF, l, r );
		l = r; lF = rF;
		}
	}

// Reduction over a time map: maximum (std::max_element semantics on finite data) and "some column descends".
PVM_HD void time_map_check( const Table & mod, int64_t f, int col, float & sec, bool & descends )
	{
	sec = mod.at( f, col );
	descends = f > 0 && !( sec >= mod.at( f - 1, col ) );
	}

} // namespace pvm
