// flan_b200/csrc/pv_generic.h -- host tables and launch interface of the any-size transform path (pv_generic_body.cuh).
#pragma once

#include <cuda_runtime.h>

#include <complex>
#include <vector>

#include "pv_generic_body.cuh"
#include "pv_policy.h"

namespace pvk {

// Largest dft size accepted (scratch per CTA grows with it: 16 bytes x 2 x the FFT length).
constexpr int GENERIC_MAX_DFT = 1 << 20;

struct GenericHost
	{
	int N = 0, even = 0, L = 0, B = 0, M = 0, bluestein = 0;
	std::vector<float2> tw, chirp, chirp_fft;
	};

// Twiddles and the Bluestein chirp, evaluated in (long) double and rounded once.
inline void generic_host_fft( std::vector<std::complex<double>> & v )     // in-place radix-2, forward, size a power of two
	{
	const size_t n = v.size();
	for( size_t i = 1, j = 0; i < n; ++i )
		{
		size_t bit = n >> 1;
		for( ; j & bit; bit >>= 1 ) j ^= bit;
		j ^= bit;
		if( i < j ) std::swap( v[i], v[j] );
		}
	const long double two_pi = 6.283185307179586476925286766559005768L;
	for( size_t len = 2; len <= n; len <<= 1 )
		{
		std::vector<std::complex<double>> w( len / 2 );
		for( size_t k = 0; k < len / 2; ++k )
			{
			const long double a = -two_pi * (long double) k / (long double) len;
			w[k] = { (double) cosl( a ), (double) sinl( a ) };
			}
		for( size_t i = 0; i < n; i += len )
			for( size_t k = 0; k < len / 2; ++k )
				{
				const std::complex<double> u = v[i + k], x = v[i + k + len / 2] * w[k];
				v[i + k] = u + x; v[i + k + len / 2] = u - x;
				}
		}
	}

inline bool build_generic( int N, GenericHost & g )
	{
	if( N < 2 || N > GENERIC_MAX_DFT ) return false;
	g.N = N; g.even = ( N % 2 == 0 ); g.L = g.even ? N / 2 : N; g.B = N / 2 + 1;
	const bool pow2 = ( g.L & ( g.L - 1 ) ) == 0;
	g.bluestein = !pow2;
	g.M = g.L;
	if( g.bluestein ) { g.M = 1; while( g.M < 2 * g.L - 1 ) g.M <<= 1; }
	const long double two_pi = 6.283185307179586476925286766559005768L, pi = two_pi / 2;
	g.tw.resize( g.M );
	for( int k = 0; k < g.M; ++k )
		{
		const long double a = -two_pi * (long double) k / (long double) g.M;
		g.tw[k].x = (float) cosl( a ); g.tw[k].y = (float) sinl( a );
		}
	g.chirp.clear(); g.chirp_fft.clear();
	if( g.bluestein )
		{
		// c[n] = e^{-i pi n^2 / L}; n^2 is reduced modulo 2L in integers so that the angle stays small and exact
		std::vector<std::complex<double>> c( g.L ), b( g.M, { 0.0, 0.0 } );
		g.chirp.resize( g.L );
		for( int n = 0; n < g.L; ++n )
			{
			const long long r = ( (long long) n * n ) % ( 2LL * g.L );
			const long double a = -pi * (long double) r / (long double) g.L;
			c[n] = { (double) cosl( a ), (double) sinl( a ) };
			g.chirp[n].x = (float) c[n].real(); g.chirp[n].y = (float) c[n].imag();
			}
		b[0] = std::conj( c[0] );
		for( int n = 1; n < g.L; ++n ) b[n] = b[g.M - n] = std::conj( c[n] );
		generic_host_fft( b );
		g.chirp_fft.resize( g.M );
		for( int k = 0; k < g.M; ++k )
			{
			g.chirp_fft[k].x = (float)( b[k].real() / g.M );
			g.chirp_fft[k].y = (float)( b[k].imag() / g.M );
			}
		}
	return true;
	}

// Geometry of a launch: threads per CTA, shared memory (0: FFT buffers in the global slab), CTAs, scratch bytes per CTA.
struct GenericGeometry { int threads; size_t smem; int64_t blocks; int64_t scratch_stride; int fft_in_smem; };
GenericGeometry generic_geometry( const GenericFft & g, int64_t state_bytes, int64_t total_segments, int sms );

cudaError_t launch_generic_analysis( const GenericAnalysisArgs & a, const GenericGeometry & geo, cudaStream_t st );
cudaError_t launch_generic_synthesis( const GenericSynthArgs & a, const GenericGeometry & geo, cudaStream_t st );

} // namespace pvk
