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
//                    (lower-frame contributions first, AudioPV.cpp:133-134);
//   PV domain    repitch per shard; stretch / modify_time with a bin-shared, non-descending map per OUTPUT shard, each
//                reading its window of input rows in place or peer-copied (multi_time); other maps gather onto device 0.
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
	            ev_done[FLAN_B200_MAX_DEVICES] = {}, ev_copied[FLAN_B200_MAX_DEVICES] = {},
	            ev_rows[FLAN_B200_MAX_DEVICES] = {};     // multi_time: input shard i's rows are written (recorded on entry)
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

// Frame ranges of a PV of F frames: cut at multiples of the whole signal's segment length; every shard at least a segment
// and at least 2 * ceil(window / hop) frames long, so that a frame's window never reaches beyond the neighbouring shard
// (fewer shards than devices for short signals).
Plan make_plan_frames( const flan_b200_multi * m, int C, int64_t F, int W, int hop, int N )
	{
	Plan p;
	p.F = F;
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

// ... of the PV that analysis makes of n samples
Plan make_plan( const flan_b200_multi * m, int C, int64_t n, int W, int hop, int N )
	{
	return make_plan_frames( m, C, flan_b200_num_frames( n, hop ), W, hop, N );
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
		for( cudaEvent_t * ev : { &m->ev_state[i], &m->ev_head[i], &m->ev_halo[i], &m->ev_done[i], &m->ev_copied[i], &m->ev_rows[i] } )
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
		for( cudaEvent_t ev : { m->ev_state[i], m->ev_head[i], m->ev_halo[i], m->ev_done[i], m->ev_copied[i], m->ev_rows[i], m->t0[i], m->t1[i] } ) if( ev ) cudaEventDestroy( ev );
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

} // extern "C"

namespace {

// flan_b200_multi_gather_pv with the handle's lock held.
int gather_pv( flan_b200_multi * m, const flan_b200_sharded_pv * pv, float * h_pv, int to, float * d_pv )
	{
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

bool strides_ok( int64_t fs, int bs, int B ) { return ( bs == 0 || bs == 1 ) && ( fs == 0 || fs == ( bs ? B : 1 ) ); }

// The header of a PV with the shape of `pv` and no rows yet.
flan_b200_sharded_pv like( const flan_b200_sharded_pv * pv )
	{
	flan_b200_sharded_pv o{};
	o.channels = pv->channels; o.frames = pv->frames; o.bins = pv->bins;
	o.sample_rate = pv->sample_rate; o.analysis_rate = pv->analysis_rate; o.window_size = pv->window_size;
	return o;
	}

// count floats of host memory -> a new block on the context's device (freed by the caller, ordered after its users).
int upload_floats( flan_b200_ctx * ctx, const float * h, int64_t count, float ** d )
	{
	int rc = flan_b200_malloc( ctx, sizeof( float ) * (size_t) count, (void **) d );
	if( !rc ) rc = flan_b200_upload( ctx, *d, h, sizeof( float ) * (size_t) count );
	return rc;
	}

// The time map of PV::stretch (factor table) or PV::modify_time (the table itself) on device i: *map and its strides.
// *owned: a block of the map's own, to be freed with the table.
int time_map_on( flan_b200_ctx * ctx, bool stretch, const float * d_table, int64_t fs, int bs, int64_t F, int B, float sr, float ar,
                 float ** map, int64_t * mfs, float ** owned )
	{
	*owned = nullptr;
	if( !stretch ) { *map = (float *) d_table; *mfs = fs; return FLAN_B200_OK; }
	const int cols = bs ? B : 1;
	int rc = flan_b200_malloc( ctx, sizeof( float ) * (size_t) F * cols, (void **) owned );
	if( !rc ) rc = flan_b200_stretch_map( ctx, d_table, fs, bs, F, B, sr, ar, *owned );       // [F][cols]: PVModify.cpp:376-382
	*map = *owned; *mfs = cols;
	return rc;
	}

// PV::stretch / PV::modify_time over the shards. A bin-shared map that never descends (the planned kernel's case) keeps
// the PV sharded: every output device computes the map and its plan for the whole signal (cheap, identical bits
// everywhere), the output is cut like an analysed PV of out_frames frames, and each output shard's segments read the
// input rows of their window -- in place when the input shard on the same device holds them, else from a staging block
// assembled by peer copies. Each shard's launch also leaves the phase summaries of its rows for
// flan_b200_multi_promise_unchanged. Anything else (a per-bin or descending map) gathers onto device 0 and runs the
// single-device path: a one-shard result.
int multi_time( flan_b200_multi * m, const flan_b200_sharded_pv * pv, bool stretch, const float * h_table, int64_t fs, int bs,
                int interp, flan_b200_sharded_pv * out )
	{
	if( !m || !pv || !h_table || !out || pv->shards < 1 || pv->shards > m->n ) return mfail( FLAN_B200_INVALID, "bad arguments" );
	const int C = pv->channels, B = pv->bins, W = pv->window_size, R = pv->shards;
	const int64_t F = pv->frames;
	const float sr = pv->sample_rate, ar = pv->analysis_rate;
	const int hop = flan_b200_hop_from_rates( sr, ar );
	if( C < 1 || B < 2 || F < 1 || hop < 1 || !( sr > 0.0f ) ) return mfail( FLAN_B200_INVALID, "bad PV format" );
	if( !strides_ok( fs, bs, B ) ) return mfail( FLAN_B200_INVALID, "table strides must be (B,1), (0,1), (1,0) or (0,0)" );
	if( interp < 0 || interp > 9 ) return mfail( FLAN_B200_INVALID, "interpolator id outside 0..9" );
	std::lock_guard<std::mutex> lock( m->call_mutex );
	*out = like( pv );
	// the point at which every input shard's rows are written: staging copies wait for this and for nothing enqueued
	// later, so no device's copies wait for another device's stretch
	for( int i = 0; i < R; ++i )
		{
		CallLock cl( m->ctx[i] );
		MCK( cudaEventRecord( m->ev_rows[i], m->ctx[i]->compute ), "event record" );
		}
	const int64_t table_count = ( fs ? F : 1 ) * ( bs ? B : 1 );
	float * d_table[FLAN_B200_MAX_DEVICES] = {}, * d_owned[FLAN_B200_MAX_DEVICES] = {}, * d_map[FLAN_B200_MAX_DEVICES] = {};
	float * d_stage[FLAN_B200_MAX_DEVICES] = {};
	int64_t * d_rows = nullptr;
	int64_t mfs = 0;
	auto cleanup = [&]()
		{
		for( int i = 0; i < m->n; ++i ) { flan_b200_free( m->ctx[i], d_table[i] ); flan_b200_free( m->ctx[i], d_owned[i] ); flan_b200_free( m->ctx[i], d_stage[i] ); }
		flan_b200_free( m->ctx[0], d_rows );
		};
	auto bail = [&]( flan_b200_ctx * ctx, int code ) { const std::string e = ctx ? flan_b200_last_error( ctx ) : thread_error(); cleanup(); flan_b200_multi_free_pv( m, out ); *out = like( pv ); return mfail( code, e ); };
	auto map_on = [&]( int i ) -> int
		{
		int rc = upload_floats( m->ctx[i], h_table, table_count, &d_table[i] );
		if( !rc ) rc = time_map_on( m->ctx[i], stretch, d_table[i], fs, bs, F, B, sr, ar, &d_map[i], &mfs, &d_owned[i] );
		return rc;
		};

	// the output frame count and the walk, from the map on device 0
	flan_b200_ctx * c0 = m->ctx[0];
	int rc = map_on( 0 );
	if( rc ) return bail( c0, rc );
	int64_t out_frames = 0; bool descends = false;
	{
		CallLock cl( c0 );
		BlockUse use( c0, { d_map[0] } );
		const pvm::Table mod{ d_map[0], mfs, bs };
		{ LaunchTimer lt( c0, 7 ); MCK( pvm::launch_map_check( mod, mfs ? F : 1, bs ? B : 1, c0->d_check, c0->sms, c0->compute ), "map check launch" ); }
		rc = read_map_check( c0, sr, hop, &out_frames, &descends );
		if( rc ) return bail( c0, rc );
	}
	out->frames = out_frames > 0 ? out_frames : 0;
	if( bs != 0 || descends || out_frames < 1 || F >= 0x7fffffff || out_frames >= 0x7fffffff )
		{
		// the single-device path on device 0, on the whole PV gathered there
		float * d_all = nullptr;
		out->shards = 1; out->frame_begin[0] = 0; out->frame_begin[1] = out->frames;
		rc = flan_b200_malloc( c0, sizeof( float ) * 2 * (size_t) C * F * B, (void **) &d_all );
		if( !rc ) rc = flan_b200_malloc( c0, sizeof( float ) * 2 * (size_t) C * std::max<int64_t>( out->frames, 1 ) * B, (void **) &out->d[0] );
		if( rc ) { flan_b200_free( c0, d_all ); return bail( c0, rc ); }
		rc = gather_pv( m, pv, nullptr, 0, d_all );
		if( rc ) { flan_b200_free( c0, d_all ); cleanup(); flan_b200_multi_free_pv( m, out ); *out = like( pv ); return rc; }
		rc = flan_b200_modify_time( c0, d_all, C, F, B, sr, ar, d_map[0], mfs, bs, interp, out_frames, out->d[0], 0 );
		flan_b200_free( c0, d_all );
		if( rc ) return bail( c0, rc );
		cleanup();
		return FLAN_B200_OK;
		}

	// output shards, cut as resynthesis will walk them
	const int N = ( B - 1 ) * 2;
	const Plan p = make_plan_frames( m, C, out_frames, W, hop, N );
	out->shards = p.shards;
	for( int j = 0; j <= p.shards; ++j ) out->frame_begin[j] = p.fb[j];
	const size_t xpos_bytes = align_up( sizeof( int ) * (size_t) F, 256 ), mix_bytes = align_up( sizeof( float ) * (size_t) out_frames, 256 );
	const size_t plan_bytes = xpos_bytes + mix_bytes + sizeof( int ) * (size_t) out_frames;
	pvm::StretchPlan plan[FLAN_B200_MAX_DEVICES] = {};
	PhaseLayout lay[FLAN_B200_MAX_DEVICES] = {};
	void * ws[FLAN_B200_MAX_DEVICES] = {};
	pvm::StretchArgs a{};
	a.F = F; a.out_frames = out_frames; a.B = B;
	a.sample_rate = sr; a.hop = float( hop ); a.interp = interp;
	// (1) map and plan of the whole signal on every output device (the workspace: phase summaries first, then the plan)
	for( int j = 0; j < p.shards; ++j )
		{
		flan_b200_ctx * ctx = m->ctx[j];
		if( j > 0 ) { rc = map_on( j ); if( rc ) return bail( ctx, rc ); }
		lay[j] = phase_layout( ctx, C, p.fb[j + 1] - p.fb[j], B, W, hop, p.seg_len );
		CallLock cl( ctx );
		BlockUse use( ctx, { d_map[j] } );
		// the whole phase layout, as flan_b200_modify_time reserves it: the resynthesis that uses these summaries finds a
		// workspace large enough, so it keeps them
		rc = get_workspace( ctx, lay[j].bytes() + plan_bytes, &ws[j] );
		if( rc ) return bail( ctx, rc );
		char * base = (char *) ws[j] + lay[j].bytes();
		plan[j] = pvm::StretchPlan{ (int *) base, (float *)( base + xpos_bytes ), (int *)( base + xpos_bytes + mix_bytes ) };
		pvm::StretchArgs aj = a;
		aj.mod = pvm::Table{ d_map[j], mfs, 0 };
		{ LaunchTimer lt( ctx, 7 ); MCK( pvm::launch_stretch_plan( aj, plan[j], ctx->compute ), "stretch plan launch" ); }
		}
	// (2) the input rows each output shard reads (one small copy from device 0)
	int64_t rows[2 * FLAN_B200_MAX_DEVICES] = {};
	{
		pvm::StretchWindows w{};
		w.n = p.shards;
		for( int j = 0; j <= p.shards; ++j ) w.xb[j] = p.fb[j];
		rc = flan_b200_malloc( c0, sizeof( rows ), (void **) &d_rows );
		if( rc ) return bail( c0, rc );
		CallLock cl( c0 );
		BlockUse use( c0, { d_rows } );
		{ LaunchTimer lt( c0, 7 ); MCK( pvm::launch_stretch_windows( plan[0], F, w, d_rows, c0->compute ), "stretch window launch" ); }
		MCK( cudaMemcpyAsync( rows, d_rows, sizeof( int64_t ) * 2 * p.shards, cudaMemcpyDeviceToHost, c0->compute ), "window read" );
		MCK( cudaStreamSynchronize( c0->compute ), "window sync" );
	}
	// (3) per output shard its row window: in place, or staged by peer copies -- all of them before any stretch launch
	DevicePlan * dp = nullptr;
	const float * rows_ptr[FLAN_B200_MAX_DEVICES] = {};
	bool staged_from[FLAN_B200_MAX_DEVICES][FLAN_B200_MAX_DEVICES] = {};
	for( int j = 0; j < p.shards; ++j )
		{
		flan_b200_ctx * ctx = m->ctx[j];
		const int64_t x0 = p.fb[j], x1 = p.fb[j + 1], r0 = rows[2 * j], r1 = rows[2 * j + 1];
		rc = flan_b200_malloc( ctx, sizeof( float ) * 2 * (size_t) C * ( x1 - x0 ) * B, (void **) &out->d[j] );
		if( rc ) return bail( ctx, rc );
		if( j < R && pv->frame_begin[j] <= r0 && r1 <= pv->frame_begin[j + 1] ) { rows_ptr[j] = pv->d[j]; continue; }
		const int64_t n_rows = r1 - r0;
		rc = flan_b200_malloc( ctx, sizeof( float ) * 2 * (size_t) C * std::max<int64_t>( n_rows, 1 ) * B, (void **) &d_stage[j] );
		if( rc ) return bail( ctx, rc );
		rows_ptr[j] = d_stage[j];
		CallLock cl( ctx );
		BlockUse use( ctx, { d_stage[j] } );
		for( int i = 0; i < R; ++i )
			{
			const int64_t lo = std::max( r0, pv->frame_begin[i] ), hi = std::min( r1, pv->frame_begin[i + 1] );
			if( hi <= lo ) continue;
			flan_b200_ctx * src = m->ctx[i];
			const int64_t src_rows = pv->frame_begin[i + 1] - pv->frame_begin[i];
			MCK( cudaStreamWaitEvent( ctx->compute, m->ev_rows[i], 0 ), "stream wait" );
			for( int c = 0; c < C; ++c )
				MCK( cudaMemcpyPeerAsync( d_stage[j] + 2 * ( (int64_t) c * n_rows + ( lo - r0 ) ) * B, ctx->device,
				                          pv->d[i] + 2 * ( (int64_t) c * src_rows + ( lo - pv->frame_begin[i] ) ) * B, src->device,
				                          sizeof( float ) * 2 * (size_t)( hi - lo ) * B, ctx->compute ), "peer copy" );
			staged_from[j][i] = true;
			}
		MCK( cudaEventRecord( m->ev_copied[j], ctx->compute ), "event record" );
		}
	// (4) per output shard its segments and their phase summaries
	for( int j = 0; j < p.shards; ++j )
		{
		flan_b200_ctx * ctx = m->ctx[j];
		const int64_t x0 = p.fb[j], x1 = p.fb[j + 1];
		rc = get_plan( ctx, N, W, hop, sr, ar, &dp );
		if( rc ) return bail( ctx, rc );
		pvm::StretchArgs aj = a;
		aj.mod = pvm::Table{ d_map[j], mfs, 0 };
		aj.out = (float2 *) out->d[j]; aj.out_row0 = x0; aj.out_channel_stride = ( x1 - x0 ) * B;
		aj.seg0 = x0 / p.seg_len;
		aj.pv = (const float2 *) rows_ptr[j];
		if( rows_ptr[j] == pv->d[j] ) { aj.row0 = pv->frame_begin[j]; aj.pv_channel_stride = ( pv->frame_begin[j + 1] - pv->frame_begin[j] ) * B; }
		else { aj.row0 = rows[2 * j]; aj.pv_channel_stride = ( rows[2 * j + 1] - rows[2 * j] ) * B; }
		CallLock cl( ctx );
		BlockUse use( ctx, { rows_ptr[j], out->d[j], d_map[j] } );
		pvm::StretchSummary summ{};
		summ.seg_len = p.seg_len; summ.segs_per_channel = lay[j].segs;
		summ.seg_out = (pvk::PhaseSeg *) ws[j];        // nothing on this context has asked for the workspace since (1)
		summ.nan_flag = ctx->summaries.nan_flag;
		summ.k = dp->host.k; summ.P = dp->host.P; summ.rcpP = dp->host.rcpP;
		MCK( cudaMemsetAsync( summ.nan_flag, 0, sizeof( int ), ctx->compute ), "flag clear" );
		{ LaunchTimer lt( ctx, 6 ); MCK( pvm::launch_stretch_segments( aj, plan[j], summ, C, ctx->compute ), "stretch launch" ); }
		ctx->summaries.publish( { out->d[j], ( x1 - x0 ) * B, x0, x1, C, B, W, lay[j].seg_len, sr, ar }, { /* needs_fix */ false, /* nan_known */ true } );
		}
	// an input shard may be freed (and its block reused) only after the copies out of it: its stream waits for them,
	// behind everything this call has enqueued there
	for( int i = 0; i < R; ++i )
		{
		CallLock cs( m->ctx[i] );
		bool read = false;
		for( int j = 0; j < p.shards; ++j )
			if( staged_from[j][i] ) { MCK( cudaStreamWaitEvent( m->ctx[i]->compute, m->ev_copied[j], 0 ), "stream wait" ); read = true; }
		if( read ) main_release( m->ctx[i], pv->d[i] );       // the block's last use is now after those waits
		}
	cleanup();
	return FLAN_B200_OK;
	}

} // namespace

extern "C" {

// PV rows of every shard -> host MF[C][F][B] (h_pv), or -> one device buffer of the same layout on device `to` (d_pv).
int flan_b200_multi_gather_pv( flan_b200_multi * m, const flan_b200_sharded_pv * pv, float * h_pv, int to, float * d_pv )
	{
	if( !m || !pv || ( !h_pv && !d_pv ) || pv->shards < 1 || pv->shards > m->n ) return mfail( FLAN_B200_INVALID, "bad arguments" );
	if( d_pv && ( to < 0 || to >= m->n ) ) return mfail( FLAN_B200_INVALID, "bad destination device" );
	std::lock_guard<std::mutex> lock( m->call_mutex );
	return gather_pv( m, pv, h_pv, to, d_pv );
	}

int flan_b200_multi_repitch( flan_b200_multi * m, const flan_b200_sharded_pv * pv, const float * h_factor,
                             int64_t factor_frame_stride, int factor_bin_stride, int interp, flan_b200_sharded_pv * pv_out )
	{
	if( !m || !pv || !h_factor || !pv_out || pv->shards < 1 || pv->shards > m->n ) return mfail( FLAN_B200_INVALID, "bad arguments" );
	const int C = pv->channels, B = pv->bins;
	if( !strides_ok( factor_frame_stride, factor_bin_stride, B ) ) return mfail( FLAN_B200_INVALID, "table strides must be (B,1), (0,1), (1,0) or (0,0)" );
	std::lock_guard<std::mutex> lock( m->call_mutex );
	*pv_out = like( pv );
	pv_out->shards = pv->shards;
	for( int i = 0; i <= pv->shards; ++i ) pv_out->frame_begin[i] = pv->frame_begin[i];
	// every frame is independent: each device repitches its own rows with its rows of the table
	for( int i = 0; i < pv->shards; ++i )
		{
		flan_b200_ctx * ctx = m->ctx[i];
		const int64_t rows = pv->frame_begin[i + 1] - pv->frame_begin[i];
		const int64_t cols = factor_bin_stride ? B : 1;
		const float * h = h_factor + pv->frame_begin[i] * factor_frame_stride;
		float * d_factor = nullptr;
		int rc = flan_b200_malloc( ctx, sizeof( float ) * 2 * (size_t) C * std::max<int64_t>( rows, 1 ) * B, (void **) &pv_out->d[i] );
		if( !rc && rows > 0 ) rc = upload_floats( ctx, h, ( factor_frame_stride ? rows : 1 ) * cols, &d_factor );
		if( !rc && rows > 0 ) rc = flan_b200_repitch( ctx, pv->d[i], C, rows, B, pv->sample_rate, d_factor, factor_frame_stride, factor_bin_stride, interp, pv_out->d[i] );
		flan_b200_free( ctx, d_factor );
		if( rc ) { const std::string e = flan_b200_last_error( ctx ); flan_b200_multi_free_pv( m, pv_out ); *pv_out = like( pv ); return mfail( rc, e ); }
		}
	return FLAN_B200_OK;
	}

int flan_b200_multi_stretch( flan_b200_multi * m, const flan_b200_sharded_pv * pv, const float * h_factor,
                             int64_t factor_frame_stride, int factor_bin_stride, int interp, flan_b200_sharded_pv * pv_out )
	{
	return multi_time( m, pv, true, h_factor, factor_frame_stride, factor_bin_stride, interp, pv_out );
	}

int flan_b200_multi_modify_time( flan_b200_multi * m, const flan_b200_sharded_pv * pv, const float * h_map_seconds,
                                 int64_t map_frame_stride, int map_bin_stride, int interp, flan_b200_sharded_pv * pv_out )
	{
	return multi_time( m, pv, false, h_map_seconds, map_frame_stride, map_bin_stride, interp, pv_out );
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
