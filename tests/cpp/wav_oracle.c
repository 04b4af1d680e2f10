/* tests/cpp/wav_oracle.c -- TEST INFRASTRUCTURE ONLY: the checker's restatement of the WAV sample conversions that
 * AudioBuffer::save / load (reference Audio/AudioBuffer.cpp:112-170) leave to libsndfile, for all six sample types
 * libsndfile writes for SF_FORMAT_WAV. libsndfile is an external dependency, not vendored in this repository
 * (version unpinned): PARITY UNPINNED. Its default conversions (normalisation on, clipping off; src/pcm.c, float32.c,
 * double64.c) are restated operation for operation, values little-endian, frames interleaved; audio is planar
 * float[C][n]. The PCM_24 case is the same restatement as oracle/pv_oracle.c pvo_pcm24_encode / _decode, which the tests
 * compare it with. tests/wav_files.py compiles this file with -ffp-contract=off (no fused multiply-add), as the oracle's
 * Makefile does. */
#include <math.h>
#include <stdint.h>
#include <string.h>

/* Bytes a value of a sub-type (libsndfile's codes: 5 PCM_U8, 2 PCM_16, 3 PCM_24, 4 PCM_32, 6 FLOAT, 7 DOUBLE) takes;
 * 0 for any other code, where encode / decode return -1. */
int wavo_pcm_width( int subtype )
	{
	switch( subtype )
		{
		case 5: return 1;
		case 2: return 2;
		case 3: return 3;
		case 4: case 6: return 4;
		case 7: return 8;
		default: return 0;
		}
	}

int wavo_pcm_encode( const float * audio, int C, int64_t n, int subtype, uint8_t * bytes )
	{
	const int width = wavo_pcm_width( subtype );
	if( !width ) return -1;
	for( int c = 0; c < C; ++c )
		for( int64_t i = 0; i < n; ++i )
			{
			float s = audio[(int64_t) c * n + i];
			s = s < -1.0f ? -1.0f : ( 1.0f < s ? 1.0f : s );               /* AudioBuffer.cpp:158-161 */
			uint8_t * o = bytes + width * ( i * C + c );                   /* AudioBuffer.cpp:153-155 */
			uint64_t v;                                                    /* little-endian value bits */
			switch( subtype )
				{
				case 5: v = (uint64_t)( lrintf( s * 127.0f ) + 128 ); break;                  /* pcm.c f2uc_array */
				case 2: v = (uint64_t) lrintf( s * 32767.0f ); break;                          /* pcm.c f2les_array */
				case 3: v = (uint64_t) lrintf( s * 8388607.0f ); break;                        /* pcm.c f2let_array */
				case 4:                                                                        /* pcm.c f2lei_array */
					/* int value = lrintf( s * 0x80000000 ): 2^31 (s = +1.0) wraps to INT_MIN; NaN is INT_MIN, SSE's
					 * 32-bit cvtss2si (the 64-bit lrintf of glibc gives LONG_MIN, whose low bits are 0) */
					v = ( s != s ) ? 0x80000000u : (uint32_t) lrintf( s * 2147483648.0f ); break;
				case 6: { uint32_t u; memcpy( &u, &s, 4 ); v = u; break; }                     /* float32.c */
				default: { const double d = (double) s; memcpy( &v, &d, 8 ); break; }          /* double64.c */
				}
			for( int k = 0; k < width; ++k ) o[k] = (uint8_t)( v >> ( 8 * k ) );
			}
	return 0;
	}

/* AudioBuffer::load (Audio/AudioBuffer.cpp:112-125): sf_readf_float of each sub-type, then de-interleave. */
int wavo_pcm_decode( const uint8_t * bytes, int C, int64_t n, int subtype, float * audio )
	{
	const int width = wavo_pcm_width( subtype );
	if( !width ) return -1;
	for( int c = 0; c < C; ++c )
		for( int64_t i = 0; i < n; ++i )
			{
			const uint8_t * b = bytes + width * ( i * C + c );
			uint64_t v = 0;
			for( int k = 0; k < width; ++k ) v |= (uint64_t) b[k] << ( 8 * k );
			float x;
			switch( subtype )
				{
				case 5: x = (float)( (int) v - 128 ) * ( 1.0f / 0x80 ); break;                                  /* pcm.c uc2f_array */
				case 2: x = (float)(int16_t) v * ( 1.0f / 0x8000 ); break;                                      /* pcm.c les2f_array */
				case 3: x = (float)(int32_t)(uint32_t)( v << 8 ) * ( 1.0f / 2147483648.0f ); break;             /* pcm.c let2f_array */
				case 4: x = (float)(int32_t)(uint32_t) v * ( 1.0f / 2147483648.0f ); break;                     /* pcm.c lei2f_array */
				case 6: { const uint32_t u = (uint32_t) v; memcpy( &x, &u, 4 ); break; }                       /* float32.c */
				default: { double d; memcpy( &d, &v, 8 ); x = (float) d; break; }                               /* double64.c */
				}
			audio[(int64_t) c * n + i] = x;
			}
	return 0;
	}
