// flan_b200/csrc/pv_core.cuh
//
// Per-thread building blocks of the phase-vocoder kernels: radix-8/4/2 Stockham FFT passes over a
// shared-memory exchange buffer, the real-FFT pack/unpack, and the float32 op sequences of the
// reference's phase_vocoder() / inverse_phase_vocoder() (reference src/flan/phase_vocoder.cpp:5-61).
//
// Everything here is __host__ __device__ and written against an `Env` (thread id, barrier, shared
// memory, async copy) so that the SAME source runs as a CUDA kernel body (pv_kernels.cu) and under
// the CPU thread emulator (emu/pv_emu.cpp, one std::thread per CUDA thread, std::barrier for
// __syncthreads). The emulator exists so index math, swizzles and barrier placement can be checked
// in a container with no GPU; it is a test harness, not a product path.
#pragma once

#include <stdint.h>
#include <math.h>
#include <string.h>
#include <vector_types.h>

#if defined(__CUDACC__)
#define PV_HD __host__ __device__ __forceinline__
#else
#define PV_HD inline
#endif

namespace pvk {

// ---------------------------------------------------------------------------------------------
// Exactly rounded float ops. nvcc contracts a*b+c into FMA by default; the reference is compiled
// without contraction, so every op of the phase-vocoder arithmetic goes through these.
// (The host build of this header is compiled with -ffp-contract=off.)
// ---------------------------------------------------------------------------------------------
PV_HD float mul_rn( float a, float b )
	{
#if defined(__CUDA_ARCH__)
	return __fmul_rn( a, b );
#else
	return a * b;
#endif
	}
PV_HD float add_rn( float a, float b )
	{
#if defined(__CUDA_ARCH__)
	return __fadd_rn( a, b );
#else
	return a + b;
#endif
	}
PV_HD float sub_rn( float a, float b )
	{
#if defined(__CUDA_ARCH__)
	return __fsub_rn( a, b );
#else
	return a - b;
#endif
	}
PV_HD float fma_rn( float a, float b, float c )
	{
#if defined(__CUDA_ARCH__)
	return __fmaf_rn( a, b, c );
#else
	return fmaf( a, b, c );
#endif
	}

// An int32 kept as the bit pattern of a float (a tensor-memory column) plus v, as such a bit pattern again.
PV_HD float int_bits_add( float bits, int v )
	{
#if defined(__CUDA_ARCH__)
	return __int_as_float( __float_as_int( bits ) + v );
#else
	int i; memcpy( &i, &bits, sizeof i );
	i = (int)( (unsigned) i + (unsigned) v );
	float r; memcpy( &r, &i, sizeof r );
	return r;
#endif
	}
PV_HD int int_bits( float bits )
	{
#if defined(__CUDA_ARCH__)
	return __float_as_int( bits );
#else
	int i; memcpy( &i, &bits, sizeof i );
	return i;
#endif
	}

// x / c for a loop-invariant divisor c with rc = RN(1/c): reciprocal multiply plus one FMA residual
// correction (Markstein). Checked exhaustively against IEEE division for every float x in
// [2^-100, 2^40] and c in { pi2, 187.5, 344.53125, 750, 375, ... } (tests/test_host_math.py samples
// it again): identical quotients. Three instructions instead of the ~10 of a generic IEEE divide.
PV_HD float div_const( float x, float c, float rc )
	{
	const float q0 = mul_rn( x, rc );
	const float e = fma_rn( -q0, c, x );
	return fma_rn( e, rc, q0 );
	}

// std::round(float): half away from zero (phase_vocoder.cpp:40).
PV_HD float round_half_away( float x )
	{
	return roundf( x );
	}

// ---------------------------------------------------------------------------------------------
// Complex helpers (float2 = re, im)
// ---------------------------------------------------------------------------------------------
PV_HD float2 cmul( float2 a, float2 w )
	{
	float2 r;
	r.x = a.x * w.x - a.y * w.y;
	r.y = a.x * w.y + a.y * w.x;
	return r;
	}

// Packed FP32x2 arithmetic (sm_100: FADD2 / FMUL2 / FFMA2 act on an aligned register pair, i.e. on one complex
// value, in ONE issue slot at the FP32 pipe's full FLOP rate). The kernels are issue-bound, so complex adds and
// lane-wise products go through these; negation is an operand modifier and costs nothing.
PV_HD float2 add2( float2 a, float2 b )
	{
#if defined(__CUDA_ARCH__)
	return __fadd2_rn( a, b );
#else
	float2 r; r.x = a.x + b.x; r.y = a.y + b.y; return r;
#endif
	}
PV_HD float2 sub2( float2 a, float2 b )
	{
#if defined(__CUDA_ARCH__)
	return __fadd2_rn( a, make_float2( -b.x, -b.y ) );
#else
	float2 r; r.x = a.x - b.x; r.y = a.y - b.y; return r;
#endif
	}
PV_HD float2 mul2( float2 a, float2 b )
	{
#if defined(__CUDA_ARCH__)
	return __fmul2_rn( a, b );
#else
	float2 r; r.x = a.x * b.x; r.y = a.y * b.y; return r;
#endif
	}
PV_HD float2 fma2( float2 a, float2 b, float2 c )
	{
#if defined(__CUDA_ARCH__)
	return __ffma2_rn( a, b, c );
#else
	float2 r; r.x = fmaf( a.x, b.x, c.x ); r.y = fmaf( a.y, b.y, c.y ); return r;
#endif
	}
PV_HD float2 splat2( float s ) { float2 r; r.x = s; r.y = s; return r; }
// Operand forms the packed instructions take for free (SASS modifiers .LO_HI, .NP, -, and scalar broadcast .F32):
PV_HD float2 swap2( float2 a ) { float2 r; r.x = a.y; r.y = a.x; return r; }     // (y, x)
PV_HD float2 np2( float2 a ) { float2 r; r.x = -a.x; r.y = a.y; return r; }      // (-x, y)
PV_HD float2 pn2( float2 a ) { float2 r; r.x = a.x; r.y = -a.y; return r; }      // (x, -y) = conj
PV_HD float2 neg2( float2 a ) { float2 r; r.x = -a.x; r.y = -a.y; return r; }
// a * w and a * conj(w) in two packed issue slots: (a.y, a.x) * w.y, then a * w.x -+ that.
PV_HD float2 cmul2( float2 a, float2 w ) { return fma2( a, splat2( w.x ), np2( mul2( swap2( a ), splat2( w.y ) ) ) ); }
PV_HD float2 cmulc2( float2 a, float2 w ) { return fma2( a, splat2( w.x ), pn2( mul2( swap2( a ), splat2( w.y ) ) ) ); }
// -i * (a - b): the rotation is done by the subtraction itself (two scalar ops, no register shuffling)
PV_HD float2 rotsub( float2 a, float2 b ) { float2 r; r.x = a.y - b.y; r.y = b.x - a.x; return r; }

// Forward 8-point DFT in place (e^{-2 pi i nk/8}); a[k] <- sum_n a[n] w^{nk}. `a` has stride S between
// elements so a radix-8 butterfly can act on a strided subset of the thread's 8 registers.
// 21 FADD2 + 10 FADD + 2 FMUL2 issue slots (52 scalar operations).
template<int S>
PV_HD void dft8( float2 * a )
	{
	const float h = 0.70710678118654752440f;
	const float2 b0 = add2( a[0*S], a[4*S] ); float2 b4 = sub2( a[0*S], a[4*S] );
	const float2 b1 = add2( a[1*S], a[5*S] ); float2 b5 = sub2( a[1*S], a[5*S] );
	const float2 b2 = add2( a[2*S], a[6*S] ); const float2 b6 = rotsub( a[2*S], a[6*S] );   // (a2 - a6) * -i
	const float2 b3 = add2( a[3*S], a[7*S] ); float2 b7 = sub2( a[3*S], a[7*S] );
	// b5 *= (1-i)/sqrt2 ; b7 *= (-1-i)/sqrt2
	float2 t;
	t.x = b5.x + b5.y; t.y = b5.y - b5.x; b5 = mul2( t, splat2( h ) );
	t.x = b7.y - b7.x; t.y = -( b7.x + b7.y ); b7 = mul2( t, splat2( h ) );
	// even outputs: DFT4 of b0..b3
	float2 c0 = add2( b0, b2 ), c2 = sub2( b0, b2 ), c1 = add2( b1, b3 ), c3 = rotsub( b1, b3 );
	a[0*S] = add2( c0, c1 ); a[4*S] = sub2( c0, c1 ); a[2*S] = add2( c2, c3 ); a[6*S] = sub2( c2, c3 );
	// odd outputs: DFT4 of b4, b5, b6, b7 (already twiddled)
	c0 = add2( b4, b6 ); c2 = sub2( b4, b6 ); c1 = add2( b5, b7 ); c3 = rotsub( b5, b7 );
	a[1*S] = add2( c0, c1 ); a[5*S] = sub2( c0, c1 ); a[3*S] = add2( c2, c3 ); a[7*S] = sub2( c2, c3 );
	}

template<int S>
PV_HD void dft4( float2 * a )
	{
	const float2 c0 = add2( a[0*S], a[2*S] ), c2 = sub2( a[0*S], a[2*S] );
	const float2 c1 = add2( a[1*S], a[3*S] ), c3 = rotsub( a[1*S], a[3*S] );
	a[0*S] = add2( c0, c1 ); a[2*S] = sub2( c0, c1 ); a[1*S] = add2( c2, c3 ); a[3*S] = sub2( c2, c3 );
	}

template<int S>
PV_HD void dft2( float2 * a )
	{
	const float2 u = a[0], v = a[S];
	a[0] = add2( u, v ); a[S] = sub2( u, v );
	}

// Multiply by the constant e^{-2 pi i K/16} = (c, s): two packed slots, the constants ride as broadcast immediates.
PV_HD float2 cmul_const( float2 v, float c, float sn )
	{
	float2 w; w.x = c; w.y = sn;
	return cmul2( v, w );
	}

// Forward 16-point DFT in place as 4 x 4 (n = j + 4m, k' = k + 4m'): inner DFT4s over m, twiddles W16^{jk}, outer
// DFT4s over j; the digit-reversed result is put back in natural order by register renaming.
template<int S>
PV_HD void dft16( float2 * a )
	{
#pragma unroll
	for( int j = 0; j < 4; ++j ) dft4<4 * S>( a + j * S );          // a[(j + 4k)S] = y_j[k]
	const float c1 = 0.92387953251128675613f, s1 = 0.38268343236508977173f, h = 0.70710678118654752440f;
	a[( 1 + 4 * 1 ) * S] = cmul_const( a[( 1 + 4 * 1 ) * S], c1, -s1 );     // W^1
	a[( 1 + 4 * 2 ) * S] = cmul_const( a[( 1 + 4 * 2 ) * S], h, -h );       // W^2
	a[( 1 + 4 * 3 ) * S] = cmul_const( a[( 1 + 4 * 3 ) * S], s1, -c1 );     // W^3
	a[( 2 + 4 * 1 ) * S] = cmul_const( a[( 2 + 4 * 1 ) * S], h, -h );       // W^2
	{ const float2 q = a[( 2 + 4 * 2 ) * S]; float2 r; r.x = q.y; r.y = -q.x; a[( 2 + 4 * 2 ) * S] = r; }   // W^4 = -i
	a[( 2 + 4 * 3 ) * S] = cmul_const( a[( 2 + 4 * 3 ) * S], -h, -h );      // W^6
	a[( 3 + 4 * 1 ) * S] = cmul_const( a[( 3 + 4 * 1 ) * S], s1, -c1 );     // W^3
	a[( 3 + 4 * 2 ) * S] = cmul_const( a[( 3 + 4 * 2 ) * S], -h, -h );      // W^6
	a[( 3 + 4 * 3 ) * S] = cmul_const( a[( 3 + 4 * 3 ) * S], -c1, s1 );     // W^9
#pragma unroll
	for( int k = 0; k < 4; ++k ) dft4<S>( a + 4 * k * S );           // a[(4k + m')S] = X[k + 4m']
	float2 o[16];
#pragma unroll
	for( int k = 0; k < 4; ++k )
#pragma unroll
		for( int m = 0; m < 4; ++m ) o[k + 4 * m] = a[( 4 * k + m ) * S];
#pragma unroll
	for( int i = 0; i < 16; ++i ) a[i * S] = o[i];
	}

// ---------------------------------------------------------------------------------------------
// FFT plan for a complex transform of M points held PT (8 or 16) per thread by T = M/PT threads.
// Passes are Stockham autosort: pass p has radix R_p and Ns_p = product of the earlier radices.
//   thread t holds, before and after every pass, the elements at logical index  t + s*T, s = 0..PT-1
//   butterfly u (u < PT/R) of thread t is jj = t + u*T and acts on registers s = u + r*(PT/R)
//   it writes element r to logical index  (jj / Ns)*Ns*R + (jj % Ns) + r*Ns
// Radix-PT passes come first (the first needs no twiddles), the remainder 2^k last.
// ---------------------------------------------------------------------------------------------
template<int M, int PT = 8> struct FftPlan
	{
	static_assert( M >= 128 && M <= 4096 && ( M & ( M - 1 ) ) == 0, "complex FFT size must be 128..4096" );
	static_assert( PT == 8 || PT == 16, "8 or 16 points per thread" );
	static constexpr int T = M / PT;
	static constexpr int log2M = ( M == 128 ) ? 7 : ( M == 256 ) ? 8 : ( M == 512 ) ? 9 : ( M == 1024 ) ? 10 : ( M == 2048 ) ? 11 : 12;
	static constexpr int log2R = ( PT == 8 ) ? 3 : 4;
	static constexpr int num_full = log2M / log2R;                // radix-PT passes
	static constexpr int last_r = 1 << ( log2M % log2R );         // 1 (none), 2, 4 or 8
	static constexpr int num_passes = num_full + ( last_r > 1 ? 1 : 0 );
	static constexpr int radix( int p ) { return p < num_full ? PT : last_r; }
	static constexpr int ns( int p ) { int n = 1; for( int i = 0; i < p; ++i ) n *= radix( i ); return n; }
	// offset (in float2) of pass p's twiddle table inside the concatenated table; pass 0 has none.
	static constexpr int tw_offset( int p ) { int o = 0; for( int i = 1; i < p; ++i ) o += ( radix( i ) - 1 ) * ns( i ); return o; }
	static constexpr int tw_total = tw_offset( num_passes );
	};

// Shared-memory exchange layouts (float2 elements; 64-bit accesses are served per half-warp, so 16 consecutive
// lanes must hit 16 distinct values of index mod 16). Padding, not XOR, so that every access of a thread is
// "per-thread base + compile-time constant" and the base is loop-invariant over the frame walk:
//   after the Ns=1 pass lanes write R*jj + r (R = 8 or 16)     -> pad(i) = i + i/16      (8t + t/2 + r | 17t + r)
//   after the Ns=8 radix-8 pass lanes write 64*(jj/8)+jj%8+8r -> pad(i) = i + 8*(i/64)  (72J + j + 8r)
//   after passes with Ns >= 16 lanes write consecutive indices -> identity
// The matching reads t + s*T are 16 consecutive, aligned indices: pad only shifts them as a block.
template<int NS> PV_HD int xpad( int i )
	{
	if( NS == 1 ) return i + ( i >> 4 );
	if( NS == 8 ) return i + ( ( i >> 6 ) << 3 );
	return i;
	}

// Exchange buffer length (float2) that covers the largest padded index.
template<int M> struct XBuf { static constexpr int size = M + M / 8; };

// One butterfly pass on the thread's PT registers: twiddle (skipped when NS == 1), DFT_R.
template<int M, int PT, int R, int NS, class TwLoad>
PV_HD void fft_butterflies( int t, float2 * v, const float2 * tw, TwLoad && ldtw )
	{
	constexpr int T = M / PT;
	constexpr int U = PT / R;           // butterflies per thread; register stride between butterfly elements
#pragma unroll
	for( int u = 0; u < U; ++u )
		{
		if( NS > 1 )
			{
			const int jm = ( t + u * T ) & ( NS - 1 );
#pragma unroll
			for( int r = 1; r < R; ++r )
				{
#ifndef PV_ABL_NOTW
				const float2 w = ldtw( tw + ( r - 1 ) * NS + jm );
#else
				float2 w; w.x = 0.5f + jm; w.y = 0.25f * r;                  // ablation build only: no table traffic
#endif
				v[u + r * U] = cmul2( v[u + r * U], w );
				}
			}
		if( R == 16 ) dft16<U>( v + u );
		if( R == 8 ) dft8<U>( v + u );
		if( R == 4 ) dft4<U>( v + u );
		if( R == 2 ) dft2<U>( v + u );
		}
	}

// The same pass with its twiddles fetched ahead of time (fft_load_twiddles before the barrier that publishes the pass's
// inputs, while the thread's value registers are dead), so the table reads' latency is not exposed behind the barrier.
template<int M, int PT, int R, int NS, class TwLoad>
PV_HD void fft_load_twiddles( int t, float2 * w, const float2 * tw, TwLoad && ldtw )
	{
	constexpr int T = M / PT, U = PT / R;
#pragma unroll
	for( int u = 0; u < U; ++u )
		{
		const int jm = ( t + u * T ) & ( NS - 1 );
#pragma unroll
		for( int r = 1; r < R; ++r ) w[u * ( R - 1 ) + r - 1] = ldtw( tw + ( r - 1 ) * NS + jm );
		}
	}
template<int M, int PT, int R, int NS>
PV_HD void fft_butterflies_w( float2 * v, const float2 * w )
	{
	constexpr int U = PT / R;
#pragma unroll
	for( int u = 0; u < U; ++u )
		{
#pragma unroll
		for( int r = 1; r < R; ++r ) v[u + r * U] = cmul2( v[u + r * U], w[u * ( R - 1 ) + r - 1] );
		if( R == 16 ) dft16<U>( v + u );
		if( R == 8 ) dft8<U>( v + u );
		if( R == 4 ) dft4<U>( v + u );
		if( R == 2 ) dft2<U>( v + u );
		}
	}

// Scatter the pass's outputs: element r of butterfly u goes to pad(expand(jj_u)) + r*NS (the pad of a butterfly's
// base does not depend on r for any of the layouts).
template<int M, int PT, int R, int NS>
PV_HD void fft_store( int t, const float2 * v, float2 * xout )
	{
	constexpr int T = M / PT;
	constexpr int U = PT / R;
#pragma unroll
	for( int u = 0; u < U; ++u )
		{
		const int jj = t + u * T;
		const int base = xpad<NS>( ( jj / NS ) * NS * R + ( jj & ( NS - 1 ) ) );
#pragma unroll
		for( int r = 0; r < R; ++r )
			xout[base + r * NS] = v[u + r * U];
		}
	}

// Gather the PT elements t + s*T written by the pass with NS: pad(t + s*T) = pad(t) + pad(s*T).
template<int M, int PT, int NS>
PV_HD void fft_load( int t, float2 * v, const float2 * xin )
	{
	constexpr int T = M / PT;
	const float2 * base = xin + xpad<NS>( t );
#pragma unroll
	for( int s = 0; s < PT; ++s )
		v[s] = base[xpad<NS>( s * T )];
	}

// ---------------------------------------------------------------------------------------------
// Phase-vocoder arithmetic
// ---------------------------------------------------------------------------------------------
struct PvConsts
	{
	float sample_rate;       // PVBuffer::Format::sample_rate
	float analysis_rate;     // float(sr) / hop                       AudioPV.cpp:25
	float rcp_analysis_rate; // RN(1 / analysis_rate)
	float pi2;               // acosf(-1) * 2.0f                      defines.h:44-45
	float rcp_pi2;           // RN(1 / pi2)
	float bin_scale;         // 1 / dft_size (exact: power of two)    PVBuffer.cpp:443-446
	int use_wrapping;        // analysis_rate < sample_rate           phase_vocoder.cpp:37
	float wrap_pi2;          // use_wrapping ? pi2 : 0 (delta - 0*round == delta: the wrap without a branch)
	};

PV_HD float rcp_approx( float x )
	{
#if defined(__CUDA_ARCH__)
	float r; asm( "rcp.approx.ftz.f32 %0, %1;" : "=f"( r ) : "f"( x ) ); return r;
#else
	return 1.0f / x;
#endif
	}
PV_HD float sqrt_approx( float x )
	{
#if defined(__CUDA_ARCH__)
	float r; asm( "sqrt.approx.ftz.f32 %0, %1;" : "=f"( r ) : "f"( x ) ); return r;
#else
	return sqrtf( x );
#endif
	}

// std::arg and std::abs of one spectrum value (phase_vocoder.cpp:43,52: atan2f and hypotf), sharing the octant
// reduction r = min/max in [0,1]:
//   phase: degree-7 minimax polynomial in r^2 (|error| < 1.2e-7 rad evaluated in float, i.e. the rounding of the
//          result) and the quadrant fix-ups; at the axes the results are the correctly rounded pi/2 and pi, and a zero
//          spectrum gives phase 0 as FFTW's exact zeros do in the reference;
//   magnitude: max * sqrt(1 + r^2), which can neither overflow nor flush to zero and is within ~4 ulp of hypotf
//          (tolerance 1e-4 relative); exact zeros give 0.
// ~23 instructions for both against ~60 for the CUDA library's atan2f + hypotf.
PV_HD float polar_pv( float re, float im, float & phase )
	{
	const float ax = fabsf( re ), ay = fabsf( im );
	const float mx = fmaxf( ax, ay );
	const float mn = fminf( ax, ay );
	const float r = mn * rcp_approx( fmaxf( mx, 1.0e-37f ) );
	const float s = r * r;
	float p = -0.00405455008149147f;
	p = fmaf( p, s, 0.021862896159291267f );
	p = fmaf( p, s, -0.055912237614393234f );
	p = fmaf( p, s, 0.09642190486192703f );
	p = fmaf( p, s, -0.1390862762928009f );
	p = fmaf( p, s, 0.19946564733982086f );
	p = fmaf( p, s, -0.33329859375953674f );
	p = fmaf( p, s, 0.9999993443489075f );
	float a = p * r;
	if( ay > ax ) a = 1.57079637050628662109375f - a;
	if( re < 0.0f ) a = 3.1415927410125732421875f - a;
	phase = copysignf( a, im );
	return mx * sqrt_approx( fmaf( r, r, 1.0f ) );
	}

// std::round(float), half away from zero (phase_vocoder.cpp:40), as trunc(x + copysign(c, x)) with c = 0.5 - 2^-25, the
// float just below one half: EXACTLY roundf for every float (checked over all 2^32 bit patterns, tools/micro/roundchk.c;
// tests/test_host_math.py samples it again). With c = 0.5 the addition itself rounds up at x = 0.5 - 2^-25 and at the odd
// integers of [2^23, 2^24); with this c a fraction >= 1/2 still carries into the next integer (the sum lies within half
// an ulp of it) and a smaller one cannot.
#define PV_ROUND_BIAS 0.49999997f
PV_HD float round_half_away_fast( float x )
	{
	return truncf( x + copysignf( PV_ROUND_BIAS, x ) );
	}

// phase_vocoder(), reference phase_vocoder.cpp:5-53, in its float32 operation order.
// `prev_phase` is the previous frame's arg() of this bin (the reference stores it in a double; it
// only ever holds a float value). Divisions by the loop constants use div_const (bit-identical).
PV_HD float2 phase_vocoder_bin( float re, float im, float & prev_phase, float bin_frequency,
                                float expected_phase_diff, const PvConsts & k )
	{
	float phase;
	float2 mf;
	mf.x = polar_pv( re, im, phase );                                       // :43 std::arg, :52 std::abs
	const float phase_diff = sub_rn( phase, prev_phase );                   // :44
	prev_phase = phase;                                                     // :45
	const float delta = sub_rn( phase_diff, expected_phase_diff );          // :48
	const float q = div_const( delta, k.pi2, k.rcp_pi2 );                   // wrap() :38-41
	const float r = round_half_away_fast( q );
	const float wrapped = k.use_wrapping ? sub_rn( delta, mul_rn( k.pi2, r ) ) : delta;    // :49
	const float df = div_const( mul_rn( wrapped, k.analysis_rate ), k.pi2, k.rcp_pi2 );   // :50
	mf.y = add_rn( bin_frequency, df );                                     // :52
	return mf;
	}

// Packed x / c, lane-wise identical to div_const.
PV_HD float2 div_const2( float2 x, float c, float rc )
	{
	const float2 q0 = mul2( x, splat2( rc ) );
	const float2 e = fma2( q0, splat2( -c ), x );
	return fma2( e, splat2( rc ), q0 );
	}

// phase_vocoder() for the two bins of a real-FFT unpack pair at once: xa = X[k], xbc = conj(X[M-k]) (the form the
// unpack produces). Lane x of every packed value belongs to bin k, lane y to bin M-k, so each arithmetic step of
// phase_vocoder.cpp:43-52 is ONE packed instruction for both bins (FADD2 / FMUL2 / FFMA2 round each lane exactly like
// their scalar forms). Lane y works on the CONJUGATE throughout: its phase, phase difference, wrap and frequency
// deviation are the exact negatives of bin M-k's (round-to-nearest, trunc and the half-away rounding are all odd
// functions), so `prev.y` holds -phase, `expd.y` must be passed as -expected_phase_diff[M-k], and the last step
// subtracts. Results are bit-identical to phase_vocoder_bin. binf = bin_to_frequency of (k, M-k). The last operation
// of each output is scalar so that (m, f) of a bin land in an adjacent register pair for the 8-byte store.
PV_HD void phase_vocoder_pair( float2 xa, float2 xbc, float2 & prev, float2 binf, float2 expd, const PvConsts & k,
                               float2 & mf_a, float2 & mf_b )
	{
	const float axa = fabsf( xa.x ), aya = fabsf( xa.y ), axb = fabsf( xbc.x ), ayb = fabsf( xbc.y );
	float2 mx, mn, rc;
	mx.x = fmaxf( axa, aya ); mn.x = fminf( axa, aya );
	mx.y = fmaxf( axb, ayb ); mn.y = fminf( axb, ayb );
	rc.x = rcp_approx( fmaxf( mx.x, 1.0e-37f ) );
	rc.y = rcp_approx( fmaxf( mx.y, 1.0e-37f ) );
	const float2 r = mul2( mn, rc );
	const float2 s = mul2( r, r );
	float2 p = fma2( splat2( -0.00405455008149147f ), s, splat2( 0.021862896159291267f ) );
	p = fma2( p, s, splat2( -0.055912237614393234f ) );
	p = fma2( p, s, splat2( 0.09642190486192703f ) );
	p = fma2( p, s, splat2( -0.1390862762928009f ) );
	p = fma2( p, s, splat2( 0.19946564733982086f ) );
	p = fma2( p, s, splat2( -0.33329859375953674f ) );
	p = fma2( p, s, splat2( 0.9999993443489075f ) );
	float2 a = mul2( p, r );
	if( aya > axa ) a.x = 1.57079637050628662109375f - a.x;
	if( xa.x < 0.0f ) a.x = 3.1415927410125732421875f - a.x;
	if( ayb > axb ) a.y = 1.57079637050628662109375f - a.y;
	if( xbc.x < 0.0f ) a.y = 3.1415927410125732421875f - a.y;
	float2 phase;
	phase.x = copysignf( a.x, xa.y );                                       // :43 std::arg of X[k]
	phase.y = copysignf( a.y, xbc.y );                                      //     -arg of X[M-k]
	const float2 q2 = fma2( r, r, splat2( 1.0f ) );
	float2 sq; sq.x = sqrt_approx( q2.x ); sq.y = sqrt_approx( q2.y );

	const float2 phase_diff = sub2( phase, prev );                          // :44
	prev = phase;                                                           // :45
	const float2 delta = sub2( phase_diff, expd );                          // :48
	const float2 q = div_const2( delta, k.pi2, k.rcp_pi2 );                 // wrap() :38-41
	float2 hf; hf.x = copysignf( PV_ROUND_BIAS, q.x ); hf.y = copysignf( PV_ROUND_BIAS, q.y );
	const float2 qh = add2( q, hf );
	float2 rr; rr.x = truncf( qh.x ); rr.y = truncf( qh.y );
	const float2 wrapped = sub2( delta, mul2( splat2( k.wrap_pi2 ), rr ) ); // :49 (wrap_pi2 = 0 when wrapping is off)
	const float2 df = div_const2( mul2( wrapped, splat2( k.analysis_rate ) ), k.pi2, k.rcp_pi2 );   // :50
	mf_a.x = mul_rn( mx.x, sq.x ); mf_a.y = add_rn( binf.x, df.x );        // :52
	mf_b.x = mul_rn( mx.y, sq.y ); mf_b.y = sub_rn( binf.y, df.y );
	}

// PVBuffer::bin_to_frequency, PVBuffer.cpp:443-446: b * float(sr) / float(dft). dft is a power of two,
// so the division is an exact scaling.
PV_HD float bin_frequency_of( int b, const PvConsts & k )
	{
	return mul_rn( mul_rn( (float) b, k.sample_rate ), k.bin_scale );
	}

// inverse_phase_vocoder(), reference phase_vocoder.cpp:55-61: float increment, double accumulator,
// wrap only when the accumulator exceeds double(pi2), modulus double(pi2) (not 2*pi).
PV_HD float phase_increment( float f, const PvConsts & k )
	{
	return mul_rn( div_const( f, k.analysis_rate, k.rcp_analysis_rate ), k.pi2 );   // :57
	}

// sinf / cosf of the accumulated phase (std::polar, phase_vocoder.cpp:60). The accumulator lives in [0, 2pi] except
// during negative excursions. Reduction to [-pi, pi] by the true 2*pi with a split constant (two FMAs: exact product,
// one rounding; accurate to ~3e-7 rad for |x| up to ~2^24 rad, beyond which float32 itself no longer resolves the
// phase), then the SFU sine / cosine (|error| ~5e-7). Measured effect on the output: 3e-7 max abs (tolerance 1e-5).
// -DPV_POLY_SINCOS selects 1-ulp polynomial kernels instead.
PV_HD void sincos_pv( float x, float * sn, float * cs )
	{
#if defined(__CUDA_ARCH__) && !defined(PV_POLY_SINCOS)
	const float k = rintf( x * 0.15915494309189535f );
	float r = fmaf( k, -6.28318548202514648f, x );
	r = fmaf( k, 1.74845553146951715e-7f, r );
	*sn = __sinf( r ); *cs = __cosf( r );
#else
	const float j = rintf( x * 0.636619772367581343f );
	float r = fmaf( j, -1.57079601287841796875f, x );
	r = fmaf( j, -3.1391647326017846353352069854736328125e-7f, r );
	r = fmaf( j, -5.390302529957764765544681040410068817436695098876953125e-15f, r );
	const int q = (int) j;
	const float s = r * r;
	float ps = fmaf( fmaf( -1.9515295891e-4f, s, 8.3321608736e-3f ), s, -1.6666654611e-1f );
	ps = fmaf( ps * s, r, r );
	float pc = fmaf( fmaf( 2.443315711809948e-5f, s, -1.388731625493765e-3f ), s, 4.166664568298827e-2f );
	pc = fmaf( pc * s, s, fmaf( -0.5f, s, 1.0f ) );
	float a = ( q & 1 ) ? pc : ps;
	float b = ( q & 1 ) ? ps : pc;
	if( q & 2 ) a = -a;
	if( ( q + 1 ) & 2 ) b = -b;
	*sn = a; *cs = b;
#endif
	}

// inverse_phase_vocoder() (phase_vocoder.cpp:55-61) for the two bins of a pack pair at once: mfk = (m, f) of bin k,
// mfm of bin M-k. The float steps (f / ar * pi2, the 2*pi reduction, m * (cos, sin)) are packed FP32x2 with lane x =
// bin k, lane y = bin M-k; the fp64 accumulate stays scalar on the FP64 pipe. Lane-wise identical to
// phase_increment + phase_accumulate + sincos_pv.
PV_HD void sincos_pv2( float2 x, float2 & sn, float2 & cs )
	{
#if defined(__CUDA_ARCH__) && !defined(PV_POLY_SINCOS)
	float2 kk = mul2( x, splat2( 0.15915494309189535f ) );
	kk.x = rintf( kk.x ); kk.y = rintf( kk.y );
	float2 r = fma2( kk, splat2( -6.28318548202514648f ), x );
	r = fma2( kk, splat2( 1.74845553146951715e-7f ), r );
	sn.x = __sinf( r.x ); cs.x = __cosf( r.x );
	sn.y = __sinf( r.y ); cs.y = __cosf( r.y );
#else
	sincos_pv( x.x, &sn.x, &cs.x );
	sincos_pv( x.y, &sn.y, &cs.y );
#endif
	}

// fmod(x, P) for x > P > 0 (exact, like libm's).
PV_HD double fmod_pos( double x, double P, double rcpP )
	{
	double n = floor( x * rcpP );
	double r = fma( -n, P, x );
	if( r < 0.0 ) r += P;
	if( r >= P ) r -= P;
	return r;
	}

// acc += inc; if( acc > P ) acc = fmod( acc, P ). The remainder is taken as x - floor(x/P)*P without the usual +-P
// fix-ups: when x/P lies within one double ulp of an integer the result can land just outside [0,P) -- congruent to
// the reference's value modulo P, i.e. the same phase to 2e-7 rad, and the next wrap re-synchronises it.
PV_HD void phase_accumulate( double & acc, float inc, double P, double rcpP )
	{
	const double x = acc + (double) inc;                                    // :58
	double r = x;
	if( x > P ) r = fma( -floor( x * rcpP ), P, x );                        // :59
	acc = r;
	}

PV_HD void inverse_pv_pair( float2 mfk, float2 mfm, double & acck, double & accm, const PvConsts & k, double P, double rcpP,
                            float2 & xk, float2 & xm )
	{
	float2 F; F.x = mfk.y; F.y = mfm.y;
	const float2 inc = mul2( div_const2( F, k.analysis_rate, k.rcp_analysis_rate ), splat2( k.pi2 ) );     // :57
	phase_accumulate( acck, inc.x, P, rcpP );                                                               // :58-59
	phase_accumulate( accm, inc.y, P, rcpP );
	float2 th; th.x = (float) acck; th.y = (float) accm;
	float2 sn, cs;
	sincos_pv2( th, sn, cs );
	float2 ek, em; ek.x = cs.x; ek.y = sn.x; em.x = cs.y; em.y = sn.y;
	xk = mul2( ek, splat2( mfk.x ) );                                                                       // :60 std::polar
	xm = mul2( em, splat2( mfm.x ) );
	}

// Split form of a plain double sum (|s| far below 2^53 * P). The remainder is rounded to a multiple of 2^-44 rad (6e-14):
// P = double(pi2_float) is a multiple of 2^-21, so from here on every sum, difference and reduction of split values is
// EXACT in double, the canonical form (q integral, r in [0,P)) of a value is unique, and combining segment summaries
// gives the same bits in any association -- a signal cut into frame-range shards (several GPUs, or slices of one launch)
// resynthesises bit for bit like the uncut signal.
PV_HD void phase_sum_from_double( double s, double P, double rcpP, double & q, double & r )
	{
	double n = floor( s * rcpP );
	double rem = fma( -n, P, s );
	if( rem < 0.0 ) { rem += P; n -= 1.0; }
	if( rem >= P ) { rem -= P; n += 1.0; }
	rem = rint( rem * 17592186044416.0 ) * 5.6843418860808015e-14;      // 2^44, 2^-44
	if( rem >= P ) { rem -= P; n += 1.0; }
	q = n; r = rem;
	}

// Running phase sum in the split form S = q*P + r, r in [0,P), q integral (held in a double): the
// reference's accumulator equals S - P*max(0, floor(max prefix of S / P)) (DESIGN.md, "phase scan"),
// so segment summaries (sum, max prefix) compose associatively.
struct PhaseSum { double q, r; };

PV_HD void phase_sum_normalize( PhaseSum & s, double P, double rcpP )
	{
	if( s.r >= P || s.r < 0.0 )
		{
		double n = floor( s.r * rcpP );
		double r = fma( -n, P, s.r );
		if( r < 0.0 ) { r += P; n -= 1.0; }
		if( r >= P ) { r -= P; n += 1.0; }
		s.r = r; s.q += n;
		}
	}

PV_HD bool phase_sum_less( const PhaseSum & a, const PhaseSum & b )
	{
	return a.q < b.q || ( a.q == b.q && a.r < b.r );
	}

struct PhaseSeg { PhaseSum sum, mx; };   // total and max prefix (the empty prefix counts as 0)

// sum.q of a summary its producer could not compute (analysis_cta<EMIT>): the scan recomputes the entry from the rows.
PV_HD double nan_marker()
	{
#if defined(__CUDA_ARCH__)
	return __longlong_as_double( 0x7ff8000000000000ll );
#else
	return (double) NAN;
#endif
	}
PV_HD bool is_nan_marker( const PhaseSeg & s ) { return s.sum.q != s.sum.q; }

// Summary of one bin over the frames of a segment, fed in frame order: total phase increment and its max prefix. Within
// a segment (a few thousand radians at most) the running sum is a plain double -- absolute error ~1e-12 rad -- and only
// the two results are converted to the split form. `bad` is the is_nan_or_inf() pre-scan of AudioPV.cpp:88. Used by
// pv_phase_seg_kernel and by every kernel that PRODUCES PV rows in frame order per bin and leaves their summary behind
// (pv_stretch_planned_kernel), so that both give the same bits.
struct PhaseSegAcc
	{
	double sum = 0.0, mx = 0.0;
	bool bad = false;
	// The running maximum only has to be taken where a non-decreasing run of prefix sums ends: right before an increment
	// that is not >= 0 (negative or NaN) and at the end. RARE_DIP: that update sits behind a real branch (a call), for
	// kernels that are short of issue slots (pv_stretch_planned_kernel: frequencies are almost never negative);
	// pv_phase_seg_kernel, which waits for HBM, lets the compiler predicate it.
#if defined(__CUDACC__)
	__host__ __device__ __noinline__
#endif
	static double dip( double sum_, double mx_ ) { return ( sum_ > mx_ ) ? sum_ : mx_; }      // by value: the accumulator stays in registers
	template<bool RARE_DIP = false>
	PV_HD void step( float2 mf, const PvConsts & k )
		{
		bad = bad || !( fabsf( mf.x ) <= 3.402823466e38f ) || !( fabsf( mf.y ) <= 3.402823466e38f );
		const float inc = phase_increment( mf.y, k );
		if( RARE_DIP ) { if( !( inc >= 0.0f ) ) mx = dip( sum, mx ); }
		else if( !( inc >= 0.0f ) ) mx = ( sum > mx ) ? sum : mx;
		sum += (double) inc;
		}
	PV_HD PhaseSeg finish( double P, double rcpP ) const
		{
		const double m = ( sum > mx ) ? sum : mx;
		PhaseSeg s;
		phase_sum_from_double( sum, P, rcpP, s.sum.q, s.sum.r );
		phase_sum_from_double( m, P, rcpP, s.mx.q, s.mx.r );
		return s;
		}
	};

} // namespace pvk
