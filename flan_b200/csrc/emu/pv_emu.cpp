// flan_b200/csrc/emu/pv_emu.cpp -- CPU thread emulator of the kernel bodies in pv_body.cuh.
//
// TEST HARNESS, not a product path: nothing in libflan_b200.so links or calls this. It runs the very
// same CTA body source the GPU runs, one std::thread per CUDA thread with std::barrier standing in for
// __syncthreads, so that index math, shared-memory layouts and barrier placement can be validated
// against the oracle in a container without a GPU (tests/test_emulator.py). libm replaces the CUDA
// math library, so results agree with the device to rounding, not bit for bit.
#include "../pv_body.cuh"
#include "../pv_tables.h"
#include "../pv_generic.h"
#include "../pv_kernel_list.h"
#include "../pv_policy.h"

#include <atomic>
#include <cmath>
#include <barrier>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <thread>
#include <vector>

using namespace pvk;

namespace {

struct HostEnv
	{
	int tid;
	std::barrier<> * bar;
	unsigned long long bulk_waits;
	std::barrier<> * warpbar;       // barrier of this thread's warp
	void sync() { bar->arrive_and_wait(); }
	void syncwarp() { warpbar->arrive_and_wait(); }
	bool any( bool p ) { return p || tid < 32; }    // used with predicates that only thread 0 raises
	float ldg( const float * p ) { return *p; }
	float2 ldg2( const float2 * p ) { return *p; }
	float4 ldg4( const float4 * p ) { return *p; }
	float2 ldcs2( const float2 * p ) { return *p; }
	void st_stream2( float2 * p, float2 v ) { *p = v; }
	void st_stream( float * p, float v ) { *p = v; }
	void red_add( float * p, float v ) { std::atomic_ref<float>( *p ).fetch_add( v ); }
	void prefetch( const void * ) {}
	void shared_add( int * p, int v ) { *p += v; }
	void cp_async8( float2 * dst, const float2 * src ) { *dst = *src; }
	void cp_async_commit() {}
	void cp_async_wait_all() {}
	// bulk copy: performed at issue, completion published through a counter (the mbarrier phase); each thread counts
	// the phases it has waited for
	typedef unsigned long long BulkBarrier;
	void bulk_init( BulkBarrier * bar ) { std::atomic_ref<BulkBarrier>( *bar ).store( 0 ); }
	void bulk_load( void * dst, const void * src, unsigned bytes, BulkBarrier * bar )
		{
		std::memcpy( dst, src, bytes );
		std::atomic_ref<BulkBarrier>( *bar ).fetch_add( 1, std::memory_order_release );
		}
	void bulk_wait( BulkBarrier * bar, unsigned )
		{
		while( std::atomic_ref<BulkBarrier>( *bar ).load( std::memory_order_acquire ) <= bulk_waits ) std::this_thread::yield();
		++bulk_waits;
		}
	// tensor memory: the CTA's 128 lanes x TMEM_COLS words, lane = thread. A stored word stays pending until the thread's
	// next tmem_wait_st; a column read before this thread wrote it, or while its store is pending, aborts.
	static constexpr int TMEM_COLS = 128;
	enum : unsigned char { TM_UNWRITTEN = 0, TM_DONE = 1, TM_PENDING = 2 };
	float * tmem_words;
	unsigned char * tmem_state;
	template<int K> void tmem_st( int col, const float * r )
		{
		for( int i = 0; i < K; ++i )
			{
			tmem_check( col + i );
			tmem_words[tid * TMEM_COLS + col + i] = r[i];
			tmem_state[tid * TMEM_COLS + col + i] = TM_PENDING;
			}
		}
	void tmem_wait_st()
		{
		for( int j = 0; j < TMEM_COLS; ++j )
			if( tmem_state[tid * TMEM_COLS + j] == TM_PENDING ) tmem_state[tid * TMEM_COLS + j] = TM_DONE;
		}
	template<int K> void tmem_ld( int col, float * r )
		{
		for( int i = 0; i < K; ++i )
			{
			tmem_check( col + i );
			const unsigned char s = tmem_state[tid * TMEM_COLS + col + i];
			if( s != TM_DONE )
				{
				std::fprintf( stderr, s == TM_PENDING ? "pv_emu: thread %d reads tensor-memory column %d while its store is pending (no tmem_wait_st since)\n"
				                                      : "pv_emu: thread %d reads tensor-memory column %d before writing it\n", tid, col + i );
				std::abort();
				}
			r[i] = tmem_words[tid * TMEM_COLS + col + i];
			}
		}
	template<int K> void tmem_wait( float * ) {}
	void tmem_check( int col )
		{
		if( tid >= 128 || col < 0 || col >= TMEM_COLS )
			{
			std::fprintf( stderr, "pv_emu: tensor-memory access of thread %d, column %d, outside the 128 lanes x %d columns\n", tid, col, TMEM_COLS );
			std::abort();
			}
		}
	};

template<int N, int PT, class Body> void run_cta( Body && body )
	{
	constexpr int T = N / ( 2 * PT );
	std::vector<float> ring( N );
	std::vector<float2> x0( XBuf<N / 2>::size ), x1( XBuf<N / 2>::size ), rowbuf( N / 2 + 16 );
	std::vector<float> tmem( 128 * HostEnv::TMEM_COLS );
	std::vector<unsigned char> tmem_state( 128 * HostEnv::TMEM_COLS, HostEnv::TM_UNWRITTEN );
	std::barrier<> bar( T );
	std::vector<std::unique_ptr<std::barrier<>>> warpbars;
	for( int w = 0; w < ( T + 31 ) / 32; ++w ) warpbars.emplace_back( new std::barrier<>( T - 32 * w < 32 ? T - 32 * w : 32 ) );
	std::vector<std::thread> th;
	for( int t = 0; t < T; ++t )
		th.emplace_back( [&, t]
			{
			HostEnv env{ t, &bar, 0, warpbars[t / 32].get(), tmem.data(), tmem_state.data() };
			body( env, ring.data(), x0.data(), x1.data(), rowbuf.data() );
			} );
	for( auto & x : th ) x.join();
	}

// The instantiation k names (PAD and EMIT as the launch policy, pv_policy.h, decides them).
template<int N, int PT> void analysis_n( const TransformKernel & k, const AnalysisArgs & a, int64_t blocks )
	{
	for( int64_t b = 0; b < blocks; ++b )
		{
		if( k.ONE )
			{
			if( k.PAD )
				run_cta<N, PT>( [&]( HostEnv & env, float *, float2 * x0, float2 * x1, float2 * ) { analysis_cta<N, PT, true, true>( a, b, env, x0, x0 ); } );
			else if( k.EMIT )      // the instantiation that also leaves the phase summaries (ring: N floats = room for the N/2 + 1 ints)
				run_cta<N, PT>( [&]( HostEnv & env, float * ring, float2 * x0, float2 * x1, float2 * ) { analysis_cta<N, PT, true, false, true>( a, b, env, x0, x0, (int *) ring ); } );
			else
				run_cta<N, PT>( [&]( HostEnv & env, float *, float2 * x0, float2 * x1, float2 * ) { analysis_cta<N, PT, true, false>( a, b, env, x0, x0 ); } );
			}
		else
			run_cta<N, PT>( [&]( HostEnv & env, float *, float2 * x0, float2 * x1, float2 * ) { analysis_cta<N, PT, false, false>( a, b, env, x0, x1 ); } );
		}
	}

template<int N> void analysis_mirror_n( const AnalysisArgs & a, int64_t blocks )
	{
	for( int64_t b = 0; b < blocks; ++b )
		run_cta<N, 16>( [&]( HostEnv & env, float * ring, float2 * x0, float2 * x1, float2 * scratch ) { analysis_cta_mirror<N>( a, b, env, x0, a.one_buffer ? x0 : x1, (float2 *) ring, scratch ); } );
	}

template<int N> void synthesis_n( const SynthArgs & a, int64_t blocks )
	{
	for( int64_t b = 0; b < blocks; ++b )
		run_cta<N, 8>( [&]( HostEnv & env, float * ola, float2 * x0, float2 * x1, float2 * rowbuf ) { if( N == 8192 ) synthesis_cta<N, true>( a, b, env, ola, x0, x0, rowbuf ); else synthesis_cta<N, false>( a, b, env, ola, x0, x1, rowbuf ); } );
	}

template<int N> void synthesis_mirror_n( const SynthArgs & a, int64_t blocks )
	{
	HostEnv::BulkBarrier bar_word = 0;
	for( int64_t b = 0; b < blocks; ++b )
		run_cta<N, 16>( [&]( HostEnv & env, float * ola, float2 * x0, float2 * x1, float2 * rowbuf )
			{
			const bool gen = !standard_shape( N, a.W, a.hop );
			if( gen ) { if( a.one_buffer ) synthesis_cta_mirror<N, true, true>( a, b, env, (float2 *) ola, x0, x0, rowbuf, &bar_word ); else synthesis_cta_mirror<N, false, true>( a, b, env, (float2 *) ola, x0, x1, rowbuf, &bar_word ); }
			else if( a.one_buffer ) synthesis_cta_mirror<N, true, false>( a, b, env, (float2 *) ola, x0, x0, rowbuf, &bar_word );
			else synthesis_cta_mirror<N, false, false>( a, b, env, (float2 *) ola, x0, x1, rowbuf, &bar_word );
			} );
	}

// The run-time-sized transform (pv_generic_body.cuh): `blocks` persistent CTAs of T threads share the segments, each
// with its slab of scratch, exactly like the device launch (pv_generic.cu) -- here one CTA after the other.
template<class Body> void run_generic_ctas( const GenericFft & g, int64_t state_bytes, int64_t blocks, int T, Body && body )
	{
	const int64_t stride = generic_align16( state_bytes + generic_fft_bytes( g ) );
	std::vector<unsigned char> scratch( (size_t)( stride * blocks ) );
	for( int64_t b = 0; b < blocks; ++b )
		{
		std::barrier<> bar( T );
		std::vector<std::thread> th;
		for( int t = 0; t < T; ++t )
			th.emplace_back( [&, t]
				{
				HostEnv env{ t, &bar, 0, nullptr };
				body( env, b, scratch.data(), stride );
				} );
		for( auto & x : th ) x.join();
		}
	}

GenericFft generic_fft_of( const GenericHost & h )
	{
	return GenericFft{ h.N, h.even, h.L, h.B, h.M, h.bluestein, h.tw.data(), h.chirp.data(), h.chirp_fft.data() };
	}

} // namespace

extern "C" {

// Same contract as flan_b200_convert_to_pv_range, on host memory. seg_len <= 0 picks the product's choice for `sms` SMs.
int pv_emu_analysis( const float * audio, int64_t audio_stride, int64_t audio_offset, int C, int64_t n_total,
                     float sr, int W, int hop, int N, int64_t frame_begin, int64_t frame_end, int seg_len, int sms,
                     float * pv_rows, int64_t pv_channel_stride, int points_per_thread, PhaseSeg * seg_out )
	{
	const bool one_buffer = points_per_thread >= 100;      // +100: the exchange buffers alias
	points_per_thread %= 100;
	const bool pt16 = points_per_thread == 16 && N >= 512;
	HostTables tb;
	if( !build_tables( N, W, hop, sr, sr / hop, tb ) ) return 1;
	const int64_t frames = frame_end - frame_begin;
	if( seg_len <= 0 ) seg_len = choose_seg_len( frames, C, sms, W, hop );
	const int segs = (int)( ( frames + seg_len - 1 ) / seg_len );
	AnalysisArgs a{};
	a.audio = audio; a.audio_stride = audio_stride; a.audio_offset = audio_offset; a.n_total = n_total;
	a.pv = (float2 *) pv_rows; a.pv_channel_stride = pv_channel_stride;
	a.frame_begin = frame_begin; a.frame_end = frame_end; a.seg_len = seg_len; a.segs_per_channel = segs;
	a.W = W; a.hop = hop;
	a.aligned2 = ( hop % 2 == 0 ) && ( ( W / 2 ) % 2 == 0 ) && ( audio_stride % 2 == 0 ) && ( audio_offset % 2 == 0 ) && ( (uintptr_t) audio % 8 == 0 );
	a.win = tb.win_analysis.data(); a.binc = tb.binc.data(); a.binc4 = tb.binc4.data(); a.post_rot = tb.post_rot.data();
	a.pass_tw = pt16 ? tb.pass_tw16.data() : tb.pass_tw.data();
	a.one_buffer = one_buffer;
	a.k = tb.k;
	a.seg_out = seg_out; a.P = tb.P; a.rcpP = tb.rcpP;
	TransformKernel k;
	k.kind = KernelKind::analysis; k.N = N; k.PT = pt16 ? 16 : 8; k.TPS = pt16 ? 512 : 768; k.ONE = pt16 && one_buffer;
	k.PAD = analysis_pad_fits( k, W, a.aligned2 );
	k.EMIT = seg_out != nullptr;
	if( k.EMIT && ( points_per_thread != 16 || !analysis_emit_fits( k, W ) ) ) return 5;
	const int64_t blocks = (int64_t) C * segs;
	if( !dft_size_is_templated( N ) )
		{
		GenericHost gh;
		if( !build_generic( N, gh ) ) return 4;
		GenericAnalysisArgs ga{};
		ga.a = a; ga.g = generic_fft_of( gh ); ga.fft_in_smem = 0; ga.total_segments = blocks;
		const int64_t ctas = blocks < 3 ? blocks : 3;          // fewer CTAs than segments: the round-robin walk is exercised
		run_generic_ctas( ga.g, generic_analysis_state_bytes( ga.g ), ctas, 24, [&]( HostEnv & env, int64_t b, unsigned char * scratch, int64_t stride )
			{
			GenericAnalysisArgs mine = ga; mine.scratch = scratch; mine.scratch_stride = stride;
			generic_analysis_cta( mine, b, ctas, 24, env, (float2 *) nullptr );
			} );
		return 0;
		}
	if( points_per_thread == 17 )       // the mirrored last pass
		{
		if( !analysis_mirror_fits( N, W, hop ) ) return 3;
		a.pass_tw = tb.pass_tw16.data();
		switch( N )
			{
			case 1024: analysis_mirror_n<1024>( a, blocks ); return 0;
			case 2048: analysis_mirror_n<2048>( a, blocks ); return 0;
			case 4096: analysis_mirror_n<4096>( a, blocks ); return 0;
			default: return 2;
			}
		}
	switch( N )
		{
		case 256: analysis_n<256, 8>( k, a, blocks ); break;
		case 512: if( pt16 ) analysis_n<512, 16>( k, a, blocks ); else analysis_n<512, 8>( k, a, blocks ); break;
		case 1024: if( pt16 ) analysis_n<1024, 16>( k, a, blocks ); else analysis_n<1024, 8>( k, a, blocks ); break;
		case 2048: if( pt16 ) analysis_n<2048, 16>( k, a, blocks ); else analysis_n<2048, 8>( k, a, blocks ); break;
		case 4096: if( pt16 ) analysis_n<4096, 16>( k, a, blocks ); else analysis_n<4096, 8>( k, a, blocks ); break;
		case 8192: if( pt16 ) analysis_n<8192, 16>( k, a, blocks ); else analysis_n<8192, 8>( k, a, blocks ); break;
		default: return 2;
		}
	return 0;
	}

// Same contract as flan_b200_convert_to_audio_range (carry_in / carry_out: [C][B] PhaseSeg, may be null).
int pv_emu_synthesis( const float * pv_rows, int64_t pv_channel_stride, int C, int64_t frame_begin, int64_t frame_end,
                      int64_t frames_total, int B, float sr, float ar, int W, int seg_len, int sms,
                      const PhaseSeg * carry_in, PhaseSeg * carry_out,
                      float * out, int64_t out_stride, int64_t out_offset, int64_t out_len, int * nan_flag, int variant )
	{
	const int N = ( B - 1 ) * 2;
	const int hop = (int)( sr / ar );
	HostTables tb;
	if( !build_tables( N, W, hop, sr, ar, tb ) ) return 1;
	const int64_t frames = frame_end - frame_begin;
	if( seg_len <= 0 ) seg_len = choose_seg_len( frames, C, sms, W, hop );
	const int segs = (int)( ( frames + seg_len - 1 ) / seg_len );
	std::vector<PhaseSeg> seg( (size_t) C * segs * B );
	std::vector<double> acc( (size_t) C * segs * B );
	int flag = 0;
	for( int c = 0; c < C; ++c )
		for( int s = 0; s < segs; ++s )
			for( int b = 0; b < B; ++b )
				{
				const int64_t fa = frame_begin + (int64_t) s * seg_len;
				const int64_t fb = fa + seg_len < frame_end ? fa + seg_len : frame_end;
				const float2 * col = (const float2 *) pv_rows + (int64_t) c * pv_channel_stride + ( fa - frame_begin ) * (int64_t) B + b;
				seg[( (size_t) c * segs + s ) * B + b] = phase_segment_summary( col, (int64_t) B, fb - fa, tb.k, tb.P, tb.rcpP, flag,
					[]( const float2 * p ) { return *p; } );
				}
	for( int c = 0; c < C; ++c )
		for( int b = 0; b < B; ++b )
			{
			PhaseSeg st; st.sum.q = st.sum.r = st.mx.q = st.mx.r = 0.0;
			if( carry_in ) st = carry_in[(size_t) c * B + b];
			for( int s = 0; s < segs; ++s )
				{
				acc[( (size_t) c * segs + s ) * B + b] = phase_state_value( st, tb.P );
				phase_state_combine( st, seg[( (size_t) c * segs + s ) * B + b], tb.P, tb.rcpP );
				}
			if( carry_out ) carry_out[(size_t) c * B + b] = st;
			}
	if( nan_flag ) *nan_flag = flag;
	if( !out ) return 0;
	for( int c = 0; c < C; ++c ) std::memset( out + (int64_t) c * out_stride, 0, sizeof( float ) * (size_t) out_len );
	SynthArgs a{};
	a.pv = (const float2 *) pv_rows; a.pv_channel_stride = pv_channel_stride;
	a.frame_begin = frame_begin; a.frame_end = frame_end;
	a.out = out; a.out_stride = out_stride; a.out_offset = out_offset;
	const int64_t total = frames_total * hop;
	a.out_lo = out_offset > 0 ? out_offset : 0;
	a.out_hi = out_offset + out_len < total ? out_offset + out_len : total;
	a.acc_start = acc.data(); a.seg_len = seg_len; a.segs_per_channel = segs;
	a.W = W; a.hop = hop; a.aligned2 = ( hop % 2 == 0 ) && ( ( W / 2 ) % 2 == 0 );
	a.win = tb.win_synthesis.data(); a.post_tw = tb.post_tw.data(); a.pass_tw = tb.pass_tw.data();
	a.pass_tw_rev = tb.pass_tw_rev.data();
	a.out_aligned2 = ( out_stride % 2 == 0 ) && ( out_offset % 2 == 0 ) && ( (uintptr_t) out % 8 == 0 );
	a.pv_aligned16 = ( (uintptr_t) pv_rows % 16 == 0 ); a.channels = C;
	a.k = tb.k; a.P = tb.P; a.rcpP = tb.rcpP;
	const int64_t blocks = (int64_t) C * segs;
	a.one_buffer = ( variant >= 100 ); variant %= 100;      // +100: one exchange buffer
	if( !dft_size_is_templated( N ) )
		{
		GenericHost gh;
		if( !build_generic( N, gh ) ) return 4;
		GenericSynthArgs ga{};
		ga.a = a; ga.g = generic_fft_of( gh ); ga.fft_in_smem = 0;
		const int64_t ctas = blocks < 3 ? blocks : 3;
		run_generic_ctas( ga.g, generic_synthesis_state_bytes( ga.g, W ), ctas, 24, [&]( HostEnv & env, int64_t b, unsigned char * scratch, int64_t stride )
			{
			GenericSynthArgs mine = ga; mine.scratch = scratch; mine.scratch_stride = stride;
			generic_synthesis_cta( mine, b, ctas, 24, env, (float2 *) nullptr );
			} );
		return 0;
		}
	if( variant == 17 )     // mirrored: the standard shape, or the general form for any aligned window and even hop
		{
		if( !synthesis_mirror_fits( N, W, hop ) ) return 3;
		switch( N )
			{
			case 1024: synthesis_mirror_n<1024>( a, blocks ); return 0;
			case 2048: synthesis_mirror_n<2048>( a, blocks ); return 0;
			case 4096: synthesis_mirror_n<4096>( a, blocks ); return 0;
			case 8192: synthesis_mirror_n<8192>( a, blocks ); return 0;
			default: return 2;
			}
		}
	switch( N )
		{
		case 256: synthesis_n<256>( a, blocks ); break;
		case 512: synthesis_n<512>( a, blocks ); break;
		case 1024: synthesis_n<1024>( a, blocks ); break;
		case 2048: synthesis_n<2048>( a, blocks ); break;
		case 4096: synthesis_n<4096>( a, blocks ); break;
		case 8192: synthesis_n<8192>( a, blocks ); break;
		default: return 2;
		}
	return 0;
	}

// What pv_phase_seg_kernel computes: the summaries of the segments of seg_len frames, [C][segs][B].
int pv_emu_phase_segments( const float * pv_rows, int C, int64_t frames, int B, float sr, float ar, int W, int seg_len, PhaseSeg * out, int * nan_flag )
	{
	const int N = ( B - 1 ) * 2;
	HostTables tb;
	if( !build_tables( N, W, (int)( sr / ar ), sr, ar, tb ) ) return 1;
	const int segs = (int)( ( frames + seg_len - 1 ) / seg_len );
	int flag = 0;
	for( int c = 0; c < C; ++c )
		for( int s = 0; s < segs; ++s )
			for( int b = 0; b < B; ++b )
				{
				const int64_t fa = (int64_t) s * seg_len, fb = fa + seg_len < frames ? fa + seg_len : frames;
				const float2 * col = (const float2 *) pv_rows + ( (int64_t) c * frames + fa ) * B + b;
				out[( (size_t) c * segs + s ) * B + b] = phase_segment_summary( col, (int64_t) B, fb - fa, tb.k, tb.P, tb.rcpP, flag, []( const float2 * p ) { return *p; } );
				}
	if( nan_flag ) *nan_flag = flag;
	return 0;
	}

// The launch policy (pv_policy.h), for tests/test_launch_policy.py: the name of the kernel choose_analysis /
// choose_synthesis return is written to out (cap bytes); returns its length, or -1 when it does not fit.
static int put_name( const std::string & s, char * out, int cap )
	{
	if( (int) s.size() >= cap ) return -1;
	std::memcpy( out, s.c_str(), s.size() + 1 );
	return (int) s.size();
	}
int pv_emu_choose_analysis( int N, int W, int hop, int C, int64_t signal_frames, int sms, int aligned2, int emit, char * out, int cap )
	{
	return put_name( choose_analysis( N, W, hop, C, signal_frames, sms, aligned2 != 0, emit != 0 ).name(), out, cap );
	}
int pv_emu_choose_synthesis( int N, int W, int hop, char * out, int cap )
	{
	return put_name( choose_synthesis( N, W, hop ).name(), out, cap );
	}
// The release kernel list (pv_kernel_list.h), one name per line.
int pv_emu_release_kernels( char * out, int cap )
	{
	std::string s;
	auto add = [&]( KernelKind kind, int N, int PT, int TPS, bool ONE, bool PAD, bool EMIT, bool GEN )
		{
		TransformKernel k;
		k.kind = kind; k.N = N; k.PT = PT; k.TPS = TPS; k.ONE = ONE; k.PAD = PAD; k.EMIT = EMIT; k.GEN = GEN;
		s += k.name() + "\n";
		};
#define PV_A( N, PT, TPS, ONE, PAD, EMIT ) add( KernelKind::analysis, N, PT, TPS, ONE, PAD, EMIT, false );
#define PV_AM( N, TPS ) add( KernelKind::analysis_mirror, N, 16, TPS, true, false, false, false );
#define PV_S( N, TPS, ONE ) add( KernelKind::synthesis, N, 8, TPS, ONE, false, false, false );
#define PV_SM( N, TPS, ONE, GEN ) add( KernelKind::synthesis_mirror, N, 16, TPS, ONE, false, false, GEN );
	PV_RELEASE_KERNELS( PV_A, PV_AM, PV_S, PV_SM )
#undef PV_A
#undef PV_AM
#undef PV_S
#undef PV_SM
	return put_name( s, out, cap );
	}

// Frames per CTA as the launch policy chooses them (pv_tables.h), for the whole-wave tests.
int pv_emu_choose_seg_len( int64_t frames, int channels, int sms, int W, int hop, int max_len, int analysis_only, int dft )
	{
	return choose_seg_len( frames, channels, sms, W, hop, max_len, analysis_only != 0, synth_ctas_per_sm( dft ) );
	}

// Host tables, for tests of the plan arithmetic.
int pv_emu_tables( int N, int W, int hop, float sr, float ar, float * win_a, float * win_s, float * expected )
	{
	HostTables tb;
	if( !build_tables( N, W, hop, sr, ar, tb ) ) return 1;
	std::memcpy( win_a, tb.win_analysis.data(), sizeof( float ) * W );
	std::memcpy( win_s, tb.win_synthesis.data(), sizeof( float ) * W );
	std::memcpy( expected, tb.expected.data(), sizeof( float ) * ( N / 2 + 1 ) );
	return 0;
	}

// round_half_away_fast against roundf on `count` floats starting at bit pattern `first`; returns mismatches (value or sign of zero).
int64_t pv_emu_round_mismatches( uint32_t first, int64_t count )
	{
	int64_t bad = 0;
	for( int64_t i = 0; i < count; ++i )
		{
		uint32_t u = first + (uint32_t) i; float x; std::memcpy( &x, &u, 4 );
		if( x != x ) continue;
		const float a = round_half_away_fast( x ), b = roundf( x );
		if( a != b || std::signbit( a ) != std::signbit( b ) ) ++bad;
		}
	return bad;
	}

// div_const against IEEE division on `count` floats starting at bit pattern `first`; returns mismatches.
int64_t pv_emu_div_const_mismatches( float c, uint32_t first, int64_t count )
	{
	const float rc = 1.0f / c;
	int64_t bad = 0;
	for( int64_t i = 0; i < count; ++i )
		{
		uint32_t u = first + (uint32_t) i; float x; std::memcpy( &x, &u, 4 );
		if( !( fabsf( x ) < 3.0e38f ) ) continue;
		if( div_const( x, c, rc ) != x / c ) ++bad;
		}
	return bad;
	}

}
