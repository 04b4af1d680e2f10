// flan_b200/csrc/pv_capi_multi.cu -- several GPUs of one box behind one handle (SURVEY 8b(1),(6), 8e; VERDICT r1 item 2).
//
// One process, one host thread, one engine context (with its own stream) per device. A signal is cut into contiguous
// frame ranges at multiples of the segment length the uncut signal would use, so every device walks exactly the
// segments a single device would, and the result is the same bit for bit:
//   analysis     each device holds its frames' samples plus a halo (window/2 + hop on the left for the phase of the frame
//                before its first, window/2 on the right); no exchange;
//   resynthesis  (1) per-bin phase state of each shard (32 * C * B bytes) copied device to device over NVLink
//                    (cudaMemcpyPeerAsync) to every later shard, combined there;
//                (2) each shard's first segment -- the frames whose windows reach into the previous shard -- is launched
//                    first; its window - hop partial sums travel to the previous device on that device's copy stream
//                    while both devices compute their interiors; the owner adds them after its own frames
//                    (lower-frame contributions first, AudioPV.cpp:133-134).
// Cross-device ordering is by CUDA events only; nothing here synchronises a device except the gather calls.
#include "pv_ctx.h"

#include <algorithm>
#include <cmath>

using namespace pvk;
using namespace pvrt;

struct flan_b200_multi
	{
	int n = 0;
	flan_b200_ctx * ctx[FLAN_B200_MAX_DEVICES] = {};
	cudaStream_t stream[FLAN_B200_MAX_DEVICES] = {};
	cudaEvent_t ev_state[FLAN_B200_MAX_DEVICES] = {}, ev_head[FLAN_B200_MAX_DEVICES] = {}, ev_halo[FLAN_B200_MAX_DEVICES] = {},
	            ev_done[FLAN_B200_MAX_DEVICES] = {}, ev_copied[FLAN_B200_MAX_DEVICES] = {};
	cudaEvent_t t0[FLAN_B200_MAX_DEVICES] = {}, t1[FLAN_B200_MAX_DEVICES] = {};     // flan_b200_multi_time_begin / _end
	int * d_nan[FLAN_B200_MAX_DEVICES] = {};      // per device: the NaN / Inf flag of the last resynthesis' pre-scan (AudioPV.cpp:88)
	bool all_peers = true;        // every pair of distinct devices has direct peer access: kernels may store into each other's memory
	std::mutex call_mutex;
	};

namespace {

thread_local std::string g_multi_error;

int mfail( int code, const std::string & msg ) { g_multi_error = msg; thread_error() = msg; return code; }

#define MCK( call, what ) do { cudaError_t e_ = ( call ); if( e_ != cudaSuccess ) return mfail( FLAN_B200_CUDA, std::string( what ) + ": " + cudaGetErrorString( e_ ) ); } while( 0 )

struct Plan
	{
	int shards = 0, seg_len = 0;
	int64_t F = 0;
	int64_t fb[FLAN_B200_MAX_DEVICES + 1] = {};
	};

// Frame ranges: cut at multiples of the whole signal's segment length; every shard at least a segment and at least
// 2 * ceil(window / hop) frames long, so that a frame's window never reaches beyond the neighbouring shard (fewer shards
// than devices for short signals).
Plan make_plan( const flan_b200_multi * m, int C, int64_t n, int W, int hop, int N )
	{
	Plan p;
	p.F = flan_b200_num_frames( n, hop );
	p.seg_len = resynthesis_seg_len( m->ctx[0], C, p.F, N, W, hop );
	const int64_t reach = 2 * (int64_t)( ( W + hop - 1 ) / hop );
	const int64_t min_frames = std::max<int64_t>( p.seg_len, ( reach + p.seg_len - 1 ) / p.seg_len * p.seg_len );
	const int64_t segs = ( p.F + p.seg_len - 1 ) / p.seg_len;
	int shards = (int) std::min<int64_t>( m->n, std::max<int64_t>( 1, p.F / min_frames ) );
	const int64_t per = ( ( segs + shards - 1 ) / shards ) * p.seg_len;
	shards = (int)( ( p.F + per - 1 ) / per );
	if( shards < 1 ) shards = 1;
	p.shards = shards;
	for( int i = 0; i <= shards; ++i ) p.fb[i] = std::min<int64_t>( p.F, per * i );
	return p;
	}

struct Span { int64_t audio_lo, audio_hi, span_lo, span_hi, own_lo, own_hi; };

Span span_of( int64_t f0, int64_t f1, int64_t F, int64_t n, int W, int hop )
	{
	Span s{};
	const int half = W / 2;
	const int64_t total = F * hop;
	if( f1 <= f0 ) return s;
	const int64_t first = f0 > 0 ? f0 - 1 : 0;
	s.audio_lo = std::max<int64_t>( 0, (int64_t) hop * first - half );
	s.audio_hi = std::max( s.audio_lo, std::min<int64_t>( n, (int64_t) hop * ( f1 - 1 ) - half + W ) );
	s.span_lo = std::max<int64_t>( 0, (int64_t) hop * f0 - half );
	s.span_hi = std::min<int64_t>( total, (int64_t) hop * ( f1 - 1 ) - half + W );
	s.own_lo = f0 == 0 ? 0 : std::min<int64_t>( total, (int64_t) hop * f0 - half + ( W - hop ) );
	s.own_hi = f1 == F ? total : std::min<int64_t>( total, (int64_t) hop * f1 - half + ( W - hop ) );
	if( s.own_lo < s.span_lo ) s.own_lo = s.span_lo;
	return s;
	}

} // namespace

extern "C" {

int flan_b200_multi_create( const int * devices, int n_devices, flan_b200_multi ** out )
	{
	if( !out ) return FLAN_B200_INVALID;
	*out = nullptr;
	int visible = flan_b200_device_count();
	if( visible < 1 ) return mfail( FLAN_B200_CUDA, "no CUDA device (flan_b200 has no CPU fallback)" );
	int ids[FLAN_B200_MAX_DEVICES];
	if( !devices )
		{
		n_devices = std::min( visible, FLAN_B200_MAX_DEVICES );
		for( int i = 0; i < n_devices; ++i ) ids[i] = i;
		}
	else
		{
		if( n_devices < 1 || n_devices > FLAN_B200_MAX_DEVICES ) return mfail( FLAN_B200_INVALID, "device list length out of range" );
		for( int i = 0; i < n_devices; ++i ) ids[i] = devices[i];
		}
	auto * m = new flan_b200_multi;
	for( int i = 0; i < n_devices; ++i )
		{
		int rc = flan_b200_create( ids[i], &m->ctx[i] );
		if( rc ) { g_multi_error = flan_b200_last_error( nullptr ); m->n = i; flan_b200_multi_destroy( m ); return rc; }
		m->n = i + 1;
		cudaSetDevice( ids[i] );
		cudaError_t e = cudaStreamCreateWithFlags( &m->stream[i], cudaStreamNonBlocking );
		for( cudaEvent_t * ev : { &m->ev_state[i], &m->ev_head[i], &m->ev_halo[i], &m->ev_done[i], &m->ev_copied[i] } )
			if( e == cudaSuccess ) e = cudaEventCreateWithFlags( ev, cudaEventDisableTiming );
		if( e == cudaSuccess ) e = cudaEventCreate( &m->t0[i] );
		if( e == cudaSuccess ) e = cudaEventCreate( &m->t1[i] );
		if( e != cudaSuccess ) { g_multi_error = cudaGetErrorString( e ); flan_b200_multi_destroy( m ); return FLAN_B200_CUDA; }
		flan_b200_set_stream( m->ctx[i], m->stream[i] );
		}
	// direct loads / stores and copies between the devices (NVLink through NVSwitch); a device listed twice, or a pair
	// without peer access, still works: the copies then go through the runtime's staging
	for( int i = 0; i < n_devices; ++i )
		for( int j = 0; j < n_devices; ++j )
			{
			if( ids[i] == ids[j] ) continue;
			int can = 0;
			if( cudaDeviceCanAccessPeer( &can, ids[i], ids[j] ) == cudaSuccess && can )
				{
				cudaSetDevice( ids[i] );
				const cudaError_t e = cudaDeviceEnablePeerAccess( ids[j], 0 );
				if( e != cudaSuccess ) { cudaGetLastError(); if( e != cudaErrorPeerAccessAlreadyEnabled ) m->all_peers = false; }
				}
			else m->all_peers = false;
			}
	*out = m;
	return FLAN_B200_OK;
	}

void flan_b200_multi_destroy( flan_b200_multi * m )
	{
	if( !m ) return;
	for( int i = 0; i < m->n; ++i )
		{
		if( !m->ctx[i] ) continue;
		cudaSetDevice( m->ctx[i]->device );
		if( m->stream[i] ) cudaStreamSynchronize( m->stream[i] );
		flan_b200_set_stream( m->ctx[i], nullptr );
		flan_b200_destroy( m->ctx[i] );
		if( m->stream[i] ) cudaStreamDestroy( m->stream[i] );
		for( cudaEvent_t ev : { m->ev_state[i], m->ev_head[i], m->ev_halo[i], m->ev_done[i], m->ev_copied[i], m->t0[i], m->t1[i] } ) if( ev ) cudaEventDestroy( ev );
		}
	delete m;
	}

const char * flan_b200_multi_last_error( const flan_b200_multi * ) { return g_multi_error.c_str(); }
int flan_b200_multi_device_count( const flan_b200_multi * m ) { return m ? m->n : 0; }
flan_b200_ctx * flan_b200_multi_ctx( flan_b200_multi * m, int i ) { return ( m && i >= 0 && i < m->n ) ? m->ctx[i] : nullptr; }

int flan_b200_multi_synchronize( flan_b200_multi * m )
	{
	if( !m ) return FLAN_B200_INVALID;
	for( int i = 0; i < m->n; ++i )
		{
		int rc = flan_b200_synchronize( m->ctx[i] );
		if( rc ) return mfail( rc, flan_b200_last_error( m->ctx[i] ) );
		}
	return FLAN_B200_OK;
	}

// Device timing across the handle: a start event on every device's stream now, and at the end the largest elapsed time
// of any device (the max over ranks of a one-process-per-GPU run).
int flan_b200_multi_time_begin( flan_b200_multi * m )
	{
	if( !m ) return FLAN_B200_INVALID;
	int rc = flan_b200_multi_synchronize( m );
	if( rc ) return rc;
	for( int i = 0; i < m->n; ++i )
		{
		cudaSetDevice( m->ctx[i]->device );
		MCK( cudaEventRecord( m->t0[i], m->stream[i] ), "event record" );
		}
	return FLAN_B200_OK;
	}

int flan_b200_multi_time_end( flan_b200_multi * m, double * ms_max )
	{
	if( !m || !ms_max ) return FLAN_B200_INVALID;
	for( int i = 0; i < m->n; ++i )
		{
		cudaSetDevice( m->ctx[i]->device );
		MCK( cudaEventRecord( m->t1[i], m->stream[i] ), "event record" );
		}
	*ms_max = 0.0;
	for( int i = 0; i < m->n; ++i )
		{
		cudaSetDevice( m->ctx[i]->device );
		MCK( cudaEventSynchronize( m->t1[i] ), "event wait" );
		float ms = 0.0f;
		MCK( cudaEventElapsedTime( &ms, m->t0[i], m->t1[i] ), "event time" );
		if( ms > *ms_max ) *ms_max = ms;
		}
	return flan_b200_multi_synchronize( m );
	}

int flan_b200_multi_plan( const flan_b200_multi * m, int channels, int64_t n, int window_size, int hop, int dft_size,
                          int * shards, int64_t * frame_begin )
	{
	if( !m || !shards || !frame_begin || hop < 1 || channels < 1 ) return FLAN_B200_INVALID;
	const Plan p = make_plan( m, channels, n, window_size, hop, dft_size );
	*shards = p.shards;
	for( int i = 0; i <= p.shards; ++i ) frame_begin[i] = p.fb[i];
	return FLAN_B200_OK;
	}

int flan_b200_multi_free_audio( flan_b200_multi * m, flan_b200_sharded_audio * a )
	{
	if( !m || !a ) return FLAN_B200_INVALID;
	for( int i = 0; i < a->shards && i < m->n; ++i ) { if( a->d[i] ) flan_b200_free( m->ctx[i], a->d[i] ); a->d[i] = nullptr; }
	a->shards = 0;
	return FLAN_B200_OK;
	}

int flan_b200_multi_free_pv( flan_b200_multi * m, flan_b200_sharded_pv * pv )
	{
	if( !m || !pv ) return FLAN_B200_INVALID;
	for( int i = 0; i < pv->shards && i < m->n; ++i ) { if( pv->d[i] ) flan_b200_free( m->ctx[i], pv->d[i] ); pv->d[i] = nullptr; }
	pv->shards = 0;
	return FLAN_B200_OK;
	}

// Host samples float[C][n] -> each device's frame range with its halos. Asynchronous for page-locked host memory.
int flan_b200_multi_scatter_audio( flan_b200_multi * m, const float * h_audio, int channels, int64_t n,
                                   int window_size, int hop, int dft_size, flan_b200_sharded_audio * out )
	{
	if( !m || !out || ( n && !h_audio ) || channels < 1 || n < 0 || hop < 1 || window_size < 2 ) return mfail( FLAN_B200_INVALID, "bad arguments" );
	std::lock_guard<std::mutex> lock( m->call_mutex );
	const Plan p = make_plan( m, channels, n, window_size, hop, dft_size );
	*out = flan_b200_sharded_audio{};
	out->channels = channels; out->n = n; out->shards = p.shards;
	for( int i = 0; i < p.shards; ++i )
		{
		const Span s = span_of( p.fb[i], p.fb[i + 1], p.F, n, window_size, hop );
		out->lo[i] = s.audio_lo; out->hi[i] = s.audio_hi;
		out->own_lo[i] = s.audio_lo; out->own_hi[i] = s.audio_hi;
		const int64_t len = s.audio_hi - s.audio_lo;
		flan_b200_ctx * ctx = m->ctx[i];
		int rc = flan_b200_malloc( ctx, sizeof( float ) * (size_t) channels * (size_t) std::max<int64_t>( len, 1 ), (void **) &out->d[i] );
		if( rc ) { flan_b200_multi_free_audio( m, out ); return mfail( rc, flan_b200_last_error( ctx ) ); }
		if( len == 0 ) continue;
		CallLock cl( ctx );
		rc = side_acquire( ctx, ctx->h2d, out->d[i] );
		if( !rc ) rc = copy_h2d_2d( ctx, out->d[i], sizeof( float ) * (size_t) len, h_audio + s.audio_lo, sizeof( float ) * (size_t) n,
		                            sizeof( float ) * (size_t) len, (size_t) channels );
		if( !rc ) rc = side_release( ctx, ctx->h2d, out->d[i] );
		if( rc ) { flan_b200_multi_free_audio( m, out ); return mfail( rc, thread_error() ); }
		}
	return FLAN_B200_OK;
	}

// Audio::convert_to_PV (AudioPV.cpp:12-78) over the shards; no exchange. pv->d[i]: MF[C][rows_i][B] on device i.
int flan_b200_multi_convert_to_pv( flan_b200_multi * m, const flan_b200_sharded_audio * a, float sample_rate,
                                   int window_size, int hop, int dft_size, flan_b200_sharded_pv * pv )
	{
	if( !m || !a || !pv || a->shards < 1 || a->shards > m->n ) return mfail( FLAN_B200_INVALID, "bad arguments" );
	std::lock_guard<std::mutex> lock( m->call_mutex );
	const Plan p = make_plan( m, a->channels, a->n, window_size, hop, dft_size );
	if( p.shards != a->shards ) return mfail( FLAN_B200_INVALID, "the audio was scattered for another window / hop / dft size" );
	const int B = dft_size / 2 + 1, C = a->channels;
	*pv = flan_b200_sharded_pv{};
	pv->channels = C; pv->frames = p.F; pv->bins = B; pv->sample_rate = sample_rate;
	pv->analysis_rate = flan_b200_analysis_rate( sample_rate, hop ); pv->window_size = window_size; pv->shards = p.shards;
	for( int i = 0; i <= p.shards; ++i ) pv->frame_begin[i] = p.fb[i];
	// flan_b200_hint_resynthesis (this thread): every shard's analysis also leaves the phase summaries of its rows, in the
	// segments of the whole signal
	const bool hint = take_resynthesis_hint();
	for( int i = 0; i < p.shards; ++i )
		{
		flan_b200_ctx * ctx = m->ctx[i];
		const int64_t rows = p.fb[i + 1] - p.fb[i];
		int rc = flan_b200_malloc( ctx, sizeof( float ) * 2 * (size_t) C * (size_t) rows * B, (void **) &pv->d[i] );
		if( !rc )
			{
			CallLock lock( ctx );
			BlockUse use( ctx, { a->d[i], pv->d[i] } );
			AnalysisCall call{ a->d[i], a->hi[i] - a->lo[i], a->lo[i], a->hi[i] - a->lo[i], C, a->n, sample_rate, window_size, hop, dft_size,
			                   p.fb[i], p.fb[i + 1], pv->d[i], rows * B };
			call.emit_summary = hint; call.emit_seg_len = p.seg_len;
			rc = analysis_range( ctx, call );
			}
		if( rc ) { const std::string e = flan_b200_last_error( ctx ); flan_b200_multi_free_pv( m, pv ); return mfail( rc, e ); }
		}
	return FLAN_B200_OK;
	}

// The two statements of a caller that resynthesises what it has just analysed (flan_b200_hint_resynthesis /
// flan_b200_promise_unchanged), for the sharded forms: per calling thread, consumed by the next
// flan_b200_multi_convert_to_pv / flan_b200_multi_convert_to_audio.
int flan_b200_multi_hint_resynthesis( flan_b200_multi * m )
	{
	if( !m ) return FLAN_B200_INVALID;
	set_resynthesis_hint();
	return FLAN_B200_OK;
	}
int flan_b200_multi_promise_unchanged( flan_b200_multi * m, const flan_b200_sharded_pv * pv )
	{
	if( !m || !pv || pv->shards < 1 ) return FLAN_B200_INVALID;
	promise_unchanged( pv->d[0] );
	return FLAN_B200_OK;
	}

// PV::convert_to_audio (AudioPV.cpp:86-139) over the shards: phase state and overlap-add halo exchanged device to device.
// out->d[i]: float[C][hi-lo], the samples [lo, hi) the frames of shard i reach; [own_lo, own_hi) of it are final.
int flan_b200_multi_convert_to_audio( flan_b200_multi * m, const flan_b200_sharded_pv * pv, flan_b200_sharded_audio * out )
	{
	if( !m || !pv || !out || pv->shards < 1 || pv->shards > m->n ) return mfail( FLAN_B200_INVALID, "bad arguments" );
	std::lock_guard<std::mutex> lock( m->call_mutex );
	const int C = pv->channels, B = pv->bins, W = pv->window_size, R = pv->shards;
	const float sr = pv->sample_rate, ar = pv->analysis_rate;
	const int hop = flan_b200_hop_from_rates( sr, ar );
	if( hop < 1 || C < 1 || B < 2 ) return mfail( FLAN_B200_INVALID, "bad PV format" );
	const int64_t F = pv->frames;
	const int seg_len = resynthesis_seg_len( m->ctx[0], C, F, ( B - 1 ) * 2, W, hop );
	for( int i = 1; i < R; ++i )
		if( pv->frame_begin[i] % seg_len != 0 ) return mfail( FLAN_B200_INVALID, "shards must begin at multiples of the signal's segment length" );
	*out = flan_b200_sharded_audio{};
	out->channels = C; out->n = F * hop; out->shards = R;
	const size_t state_bytes = sizeof( PhaseSeg ) * (size_t) C * B;
	PhaseSeg * d_state[FLAN_B200_MAX_DEVICES] = {}, * d_all[FLAN_B200_MAX_DEVICES] = {}, * d_carry[FLAN_B200_MAX_DEVICES] = {};
	float * d_halo[FLAN_B200_MAX_DEVICES] = {};
	Span sp[FLAN_B200_MAX_DEVICES];
	int rc = FLAN_B200_OK;
	auto cleanup = [&]( bool failed )
		{
		// scratch goes back to each device's block cache (ordered after the work enqueued above)
		for( int i = 0; i < R; ++i )
			{
			flan_b200_free( m->ctx[i], d_state[i] ); flan_b200_free( m->ctx[i], d_all[i] );
			flan_b200_free( m->ctx[i], d_carry[i] ); flan_b200_free( m->ctx[i], d_halo[i] );
			}
		if( failed ) flan_b200_multi_free_audio( m, out );
		};
	auto bail = [&]( flan_b200_ctx * ctx, int code ) { const std::string e = ctx ? flan_b200_last_error( ctx ) : thread_error(); cleanup( true ); return mfail( code, e ); };

	const bool unchanged = take_promise( pv->d[0] );       // flan_b200_promise_unchanged( ., pv->d[0] ) by this thread
	// (0) where the states of the earlier shards will land on each later device
	for( int i = 1; i < R; ++i )
		{
		flan_b200_ctx * ctx = m->ctx[i];
		rc = flan_b200_malloc( ctx, state_bytes * i, (void **) &d_all[i] );
		if( !rc ) rc = flan_b200_malloc( ctx, state_bytes, (void **) &d_carry[i] );
		if( rc ) return bail( ctx, rc );
		CallLock cl( ctx );
		BlockUse use( ctx, { d_all[i] } );                  // earlier users of the recycled block are ahead of this point on the stream
		MCK( cudaEventRecord( m->ev_copied[i], ctx->compute ), "event record" );
		}
	// (1) phase state of every shard, on its device; one kernel then pushes it to every later device (peer stores)
	for( int i = 0; i < R; ++i )
		{
		flan_b200_ctx * ctx = m->ctx[i];
		sp[i] = span_of( pv->frame_begin[i], pv->frame_begin[i + 1], F, out->n, W, hop );
		rc = flan_b200_malloc( ctx, state_bytes, (void **) &d_state[i] );
		if( rc ) return bail( ctx, rc );
		CallLock cl( ctx );
		BlockUse use( ctx, { pv->d[i], d_state[i] } );
		const int64_t rows = pv->frame_begin[i + 1] - pv->frame_begin[i];
		SynthCall s{ pv->d[i], rows * B, C, pv->frame_begin[i], pv->frame_begin[i + 1], F, B, sr, ar, W };
		s.d_carry_out = d_state[i]; s.summary_only = true; s.seg_len = seg_len;
		s.reuse_summary = unchanged;      // summaries the shard's analysis left (flan_b200_hint_resynthesis), if they are still this buffer's
		m->d_nan[i] = ctx->d_flags + ( ctx->flag_next++ % flan_b200_ctx::FLAG_SLOTS );
		MCK( cudaMemsetAsync( m->d_nan[i], 0, sizeof( int ), ctx->compute ), "flag clear" );
		s.d_nan_flag = m->d_nan[i];
		rc = synth_range( ctx, s );
		if( rc ) return bail( ctx, rc );
		if( i + 1 < R && m->all_peers )
			{
			pvk::StatePush push{};
			push.src = (const uint4 *) d_state[i]; push.n16 = (unsigned)( state_bytes / 16 );
			int n = 0;
			for( int j = i + 1; j < R; ++j, ++n )
				{
				MCK( cudaStreamWaitEvent( ctx->compute, m->ev_copied[j], 0 ), "stream wait" );
				push.dst[n] = (uint4 *)( (char *) d_all[j] + state_bytes * i );
				}
			MCK( pvk::launch_state_push( push, n, ctx->compute ), "state push launch" );
			ctx->launches++;
			}
		MCK( cudaEventRecord( m->ev_state[i], ctx->compute ), "event record" );
		}
	// (2) ... and are combined there
	for( int i = 1; i < R; ++i )
		{
		flan_b200_ctx * ctx = m->ctx[i];
		CallLock cl( ctx );
		for( int q = 0; q < i; ++q )
			{
			MCK( cudaStreamWaitEvent( ctx->compute, m->ev_state[q], 0 ), "stream wait" );
			// without peer access everywhere the runtime stages the copies
			if( !m->all_peers ) MCK( cudaMemcpyPeerAsync( (char *) d_all[i] + state_bytes * q, ctx->device, d_state[q], m->ctx[q]->device, state_bytes, ctx->compute ), "peer copy" );
			}
		if( !m->all_peers ) MCK( cudaEventRecord( m->ev_done[i], ctx->compute ), "event record" );
		rc = flan_b200_phase_carry( ctx, (const flan_b200_phase_state *) d_all[i], i, C, B, (flan_b200_phase_state *) d_carry[i] );
		if( rc ) return bail( ctx, rc );
		}
	// (3) transforms: the first segment of every shard first, then its halo leaves while the rest computes
	const int64_t ov_max = std::max( 0, W - hop );
	for( int i = 0; i < R; ++i )
		{
		flan_b200_ctx * ctx = m->ctx[i];
		const int64_t len = sp[i].span_hi - sp[i].span_lo;
		out->lo[i] = sp[i].span_lo; out->hi[i] = sp[i].span_hi; out->own_lo[i] = sp[i].own_lo; out->own_hi[i] = sp[i].own_hi;
		rc = flan_b200_malloc( ctx, sizeof( float ) * (size_t) C * (size_t) std::max<int64_t>( len, 1 ), (void **) &out->d[i] );
		if( !rc && i + 1 < R ) rc = flan_b200_malloc( ctx, sizeof( float ) * (size_t) C * (size_t) std::max<int64_t>( ov_max, 1 ), (void **) &d_halo[i] );
		if( rc ) return bail( ctx, rc );
		CallLock cl( ctx );
		BlockUse use( ctx, { pv->d[i], out->d[i], d_carry[i] } );
		const int64_t rows = pv->frame_begin[i + 1] - pv->frame_begin[i];
		SynthCall s{ pv->d[i], rows * B, C, pv->frame_begin[i], pv->frame_begin[i + 1], F, B, sr, ar, W };
		s.d_carry_in = d_carry[i]; s.reuse_summary = true; s.seg_len = seg_len;
		s.d_out = out->d[i]; s.out_stride = len; s.out_offset = sp[i].span_lo; s.out_len = len;
		if( i > 0 )
			{
			s.head_segments = 1;        // seg_len * hop >= window - hop: the first segment holds every frame that reaches shard i-1
			s.head_event = m->ev_head[i];
			}
		rc = synth_range( ctx, s );
		if( rc ) return bail( ctx, rc );
		}
	// (4) halo: samples [span_lo, own_lo) of shard i+1 are partial sums owned by shard i
	for( int i = 0; i + 1 < R; ++i )
		{
		flan_b200_ctx * ctx = m->ctx[i], * nxt = m->ctx[i + 1];
		const int64_t h_lo = sp[i + 1].span_lo, h_hi = std::min( sp[i + 1].own_lo, sp[i + 1].span_hi );
		const int64_t hn = h_hi - h_lo;
		if( hn <= 0 ) continue;
		CallLock cl( ctx );
		const int64_t nlen = sp[i + 1].span_hi - sp[i + 1].span_lo, len = sp[i].span_hi - sp[i].span_lo;
		MCK( cudaStreamWaitEvent( ctx->h2d, m->ev_head[i + 1], 0 ), "copy stream wait" );
		for( int c = 0; c < C; ++c )
			MCK( cudaMemcpyPeerAsync( d_halo[i] + (int64_t) c * hn, ctx->device, out->d[i + 1] + (int64_t) c * nlen, nxt->device,
			                          sizeof( float ) * (size_t) hn, ctx->h2d ), "peer copy" );
		MCK( cudaEventRecord( m->ev_halo[i], ctx->h2d ), "event record" );
		MCK( cudaStreamWaitEvent( ctx->compute, m->ev_halo[i], 0 ), "stream wait" );
		if( h_lo < sp[i].span_lo || h_hi > sp[i].span_hi ) return bail( nullptr, mfail( FLAN_B200_INVALID, "internal: halo outside the owner's span" ) );
		for( int c = 0; c < C; ++c )
			{
			rc = flan_b200_add( ctx, out->d[i] + (int64_t) c * len + ( h_lo - sp[i].span_lo ), d_halo[i] + (int64_t) c * hn, hn );
			if( rc ) return bail( ctx, rc );
			}
		// the neighbour must not recycle its span before the copy above has run: its stream waits for it
			{
			CallLock cn( nxt );
			MCK( cudaStreamWaitEvent( nxt->stream, m->ev_halo[i], 0 ), "stream wait" );
			}
		}
	// (staged copies only) the state of shard q was read by the streams of the later devices: its block may only be
	// recycled after those copies
	if( !m->all_peers )
		for( int q = 0; q + 1 < R; ++q )
			{
			CallLock cl( m->ctx[q] );
			for( int i = q + 1; i < R; ++i ) MCK( cudaStreamWaitEvent( m->ctx[q]->compute, m->ev_done[i], 0 ), "stream wait" );
			main_release( m->ctx[q], d_state[q] );
			}
	cleanup( false );
	return FLAN_B200_OK;
	}

// Final samples of every shard -> host float[C][n_out]. Returns once the bytes have arrived.
int flan_b200_multi_gather_audio( flan_b200_multi * m, const flan_b200_sharded_audio * a, float * h_audio )
	{
	if( !m || !a || !h_audio || a->shards < 1 || a->shards > m->n ) return mfail( FLAN_B200_INVALID, "bad arguments" );
	std::lock_guard<std::mutex> lock( m->call_mutex );
	for( int i = 0; i < a->shards; ++i )
		{
		flan_b200_ctx * ctx = m->ctx[i];
		const int64_t cnt = a->own_hi[i] - a->own_lo[i], len = a->hi[i] - a->lo[i];
		if( cnt <= 0 ) continue;
		CallLock cl( ctx );
		int rc = side_acquire( ctx, ctx->d2h, a->d[i] );
		// foreign to the block history: the transforms ran on this context's stream, order the copy after them
		if( !rc ) { MCK( cudaEventRecord( m->ev_done[i], ctx->compute ), "event record" ); MCK( cudaStreamWaitEvent( ctx->d2h, m->ev_done[i], 0 ), "copy stream wait" ); }
		if( !rc ) rc = copy_d2h_2d( ctx, h_audio + a->own_lo[i], sizeof( float ) * (size_t) a->n, a->d[i] + ( a->own_lo[i] - a->lo[i] ),
		                            sizeof( float ) * (size_t) len, sizeof( float ) * (size_t) cnt, (size_t) a->channels );
		if( !rc ) rc = side_release( ctx, ctx->d2h, a->d[i] );
		if( rc ) return mfail( rc, thread_error() );
		}
	for( int i = 0; i < a->shards; ++i )
		{
		int rc = flan_b200_wait_copies( m->ctx[i], a->d[i] );
		if( rc ) return mfail( rc, flan_b200_last_error( m->ctx[i] ) );
		}
	return FLAN_B200_OK;
	}

// PV rows of every shard -> host MF[C][F][B] (h_pv), or -> one device buffer of the same layout on device `to` (d_pv).
int flan_b200_multi_gather_pv( flan_b200_multi * m, const flan_b200_sharded_pv * pv, float * h_pv, int to, float * d_pv )
	{
	if( !m || !pv || ( !h_pv && !d_pv ) || pv->shards < 1 || pv->shards > m->n ) return mfail( FLAN_B200_INVALID, "bad arguments" );
	if( d_pv && ( to < 0 || to >= m->n ) ) return mfail( FLAN_B200_INVALID, "bad destination device" );
	std::lock_guard<std::mutex> lock( m->call_mutex );
	const int C = pv->channels, B = pv->bins;
	const int64_t F = pv->frames;
	for( int i = 0; i < pv->shards; ++i )
		{
		flan_b200_ctx * ctx = m->ctx[i];
		const int64_t rows = pv->frame_begin[i + 1] - pv->frame_begin[i];
		if( rows <= 0 ) continue;
		const size_t width = sizeof( float ) * 2 * (size_t) rows * B;
		CallLock cl( ctx );
		MCK( cudaEventRecord( m->ev_done[i], ctx->compute ), "event record" );
		if( h_pv )
			{
			int rc = side_acquire( ctx, ctx->d2h, pv->d[i] );
			MCK( cudaStreamWaitEvent( ctx->d2h, m->ev_done[i], 0 ), "copy stream wait" );
			if( !rc ) rc = copy_d2h_2d( ctx, h_pv + 2 * pv->frame_begin[i] * B, sizeof( float ) * 2 * (size_t) F * B, pv->d[i], width, width, (size_t) C );
			if( !rc ) rc = side_release( ctx, ctx->d2h, pv->d[i] );
			if( rc ) return mfail( rc, thread_error() );
			}
		if( d_pv )
			{
			flan_b200_ctx * dst = m->ctx[to];
			CallLock cd( dst );
			dst->summaries.drop();      // new rows in d_pv, written without the workspace
			MCK( cudaStreamWaitEvent( dst->stream, m->ev_done[i], 0 ), "stream wait" );
			for( int c = 0; c < C; ++c )
				MCK( cudaMemcpyPeerAsync( d_pv + 2 * ( (int64_t) c * F + pv->frame_begin[i] ) * B, dst->device,
				                          pv->d[i] + 2 * (int64_t) c * rows * B, ctx->device, width, dst->stream ), "peer copy" );
			// the source shard may be freed (and its block reused) only after the copy: its stream waits for the destination's
			// (an event is recorded on a stream of its own device: the destination's)
			MCK( cudaEventRecord( m->ev_copied[to], dst->stream ), "event record" );
			MCK( cudaStreamWaitEvent( ctx->compute, m->ev_copied[to], 0 ), "stream wait" );
			}
		}
	if( h_pv )
		for( int i = 0; i < pv->shards; ++i )
			{
			int rc = flan_b200_wait_copies( m->ctx[i], pv->d[i] );
			if( rc ) return mfail( rc, flan_b200_last_error( m->ctx[i] ) );
			}
	return FLAN_B200_OK;
	}

// Host-buffer forms: what flan::Audio::convert_to_PV / flan::PV::convert_to_audio call for long signals.
int flan_b200_multi_convert_to_pv_host( flan_b200_multi * m, const float * h_audio, int channels, int64_t n, float sample_rate,
                                        int window_size, int hop, int dft_size, flan_b200_sharded_pv * pv )
	{
	flan_b200_sharded_audio a{};
	int rc = flan_b200_multi_scatter_audio( m, h_audio, channels, n, window_size, hop, dft_size, &a );
	if( rc ) return rc;
	rc = flan_b200_multi_convert_to_pv( m, &a, sample_rate, window_size, hop, dft_size, pv );
	flan_b200_multi_free_audio( m, &a );        // back to the block caches, ordered after the transforms
	return rc;
	}

int flan_b200_multi_convert_to_audio_host( flan_b200_multi * m, const flan_b200_sharded_pv * pv, float * h_audio_out, int * nan_or_inf )
	{
	flan_b200_sharded_audio a{};
	int rc = flan_b200_multi_convert_to_audio( m, pv, &a );
	if( rc ) return rc;
	rc = flan_b200_multi_gather_audio( m, &a, h_audio_out );
	if( !rc && nan_or_inf )
		{
		// the gather above waited for every shard's transform: the pre-scan flags are final
		*nan_or_inf = 0;
		for( int i = 0; i < a.shards; ++i )
			{
			int f = 0;
			cudaSetDevice( m->ctx[i]->device );
			MCK( cudaMemcpy( &f, m->d_nan[i], sizeof( int ), cudaMemcpyDeviceToHost ), "flag read" );
			*nan_or_inf |= f;
			}
		}
	flan_b200_multi_free_audio( m, &a );
	return rc;
	}

} // extern "C"
