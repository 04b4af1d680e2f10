// flan_b200/csrc/pv_capi.cu -- the C ABI declared in include/flan_b200.h: context, device blocks, the two transforms in
// their device-pointer, frame-range and pipelined host-buffer forms. (PV-domain chain: pv_capi_modify.cu; file formats:
// pv_capi_io.cu; several GPUs: pv_capi_multi.cu.)
//
// Host-side orchestration only: plan (constant table) cache, scratch workspace, launch geometry, stream ordering and
// error mapping. All arithmetic of the path runs in the kernels of pv_kernels.cu / pv_generic.cu; there is no CPU
// fallback here -- every entry point fails with FLAN_B200_CUDA when no device is usable.
#include "pv_ctx.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>

using namespace pvk;
using namespace pvrt;

static_assert( sizeof( flan_b200_phase_state ) == sizeof( PhaseSeg ), "phase state layout" );

// ------------------------------------------------------------------------------------------------------------------
// runtime pieces shared with the other pv_capi*.cu files (declared in pv_ctx.h)
// ------------------------------------------------------------------------------------------------------------------
namespace pvrt {

std::string & thread_error()
	{
	thread_local std::string e;
	return e;
	}

int fail( flan_b200_ctx *, int code, const std::string & msg )
	{
	thread_error() = msg;
	return code;
	}

int cuda_fail( flan_b200_ctx * ctx, cudaError_t e, const char * what )
	{
	return fail( ctx, e == cudaErrorMemoryAllocation ? FLAN_B200_NOMEM : FLAN_B200_CUDA,
	             std::string( what ) + ": " + cudaGetErrorString( e ) );
	}

// ---- copy threads --------------------------------------------------------------------------------------------
CopyPool::CopyPool( int threads )
	{
	for( int i = 1; i < threads; ++i ) workers_.emplace_back( [this] { run(); } );
	}

CopyPool::~CopyPool()
	{
		{ std::lock_guard<std::mutex> l( m_ ); stop_ = true; }
	cv_.notify_all();
	for( auto & t : workers_ ) t.join();
	}

void CopyPool::run()
	{
	for( ;; )
		{
		Task task;
			{
			std::unique_lock<std::mutex> l( m_ );
			cv_.wait( l, [this] { return stop_ || !queue_.empty(); } );
			if( queue_.empty() ) return;
			task = queue_.back(); queue_.pop_back();
			}
		std::memcpy( task.dst, task.src, task.bytes );
			{
			std::lock_guard<std::mutex> l( m_ );
			if( --outstanding_ == 0 ) done_cv_.notify_all();
			}
		}
	}

void CopyPool::copy( void * dst, const void * src, size_t bytes )
	{
	const int parts = threads();
	const size_t per = align_up( ( bytes + parts - 1 ) / parts, 4096 );
	if( parts == 1 || bytes < ( size_t( 256 ) << 10 ) ) { std::memcpy( dst, src, bytes ); return; }
	size_t mine = 0;
		{
		std::lock_guard<std::mutex> l( m_ );
		for( int i = 0; i < parts; ++i )
			{
			const size_t lo = per * i, hi = std::min( bytes, lo + per );
			if( lo >= hi ) break;
			if( i == 0 ) { mine = hi; continue; }
			queue_.push_back( { (char *) dst + lo, (const char *) src + lo, hi - lo } );
			++outstanding_;
			}
		}
	cv_.notify_all();
	std::memcpy( dst, src, mine );
	std::unique_lock<std::mutex> l( m_ );
	done_cv_.wait( l, [this] { return outstanding_ == 0; } );
	}

CopyPool & copy_pool( flan_b200_ctx * ctx )
	{
	if( !ctx->copy_pool )
		{
		const unsigned hw = std::thread::hardware_concurrency();
		ctx->copy_pool.reset( new CopyPool( (int) std::max( 1u, std::min( 4u, hw / 2 ) ) ) );
		}
	return *ctx->copy_pool;
	}

// ---- plans ----------------------------------------------------------------------------------------------------
template<class T> static cudaError_t upload_vec( const std::vector<T> & v, T ** d, cudaStream_t st )
	{
	cudaError_t e = cudaMalloc( (void **) d, sizeof( T ) * ( v.empty() ? 1 : v.size() ) );
	if( e != cudaSuccess ) return e;
	if( v.empty() ) return cudaSuccess;
	// pageable source: the copy is staged before the call returns, so `v` may die afterwards
	return cudaMemcpyAsync( *d, v.data(), sizeof( T ) * v.size(), cudaMemcpyHostToDevice, st );
	}

void free_plan( DevicePlan * p )
	{
	cudaFree( p->win_analysis ); cudaFree( p->win_synthesis ); cudaFree( p->expected ); cudaFree( p->binc );
	cudaFree( p->post_tw ); cudaFree( p->post_rot ); cudaFree( p->binc4 ); cudaFree( p->pass_tw ); cudaFree( p->pass_tw16 );
	cudaFree( p->pass_tw_rev );
	cudaFree( p->g_tw ); cudaFree( p->g_chirp ); cudaFree( p->g_chirp_fft );
	}

int get_plan( flan_b200_ctx * ctx, int N, int W, int hop, float sr, float ar, DevicePlan ** out )
	{
	if( N < 2 || N > GENERIC_MAX_DFT )
		return fail( ctx, FLAN_B200_UNSUPPORTED, "dft_size must lie in [2, " + std::to_string( GENERIC_MAX_DFT ) + "], got " + std::to_string( N ) );
	if( W < 2 || W > N || hop < 1 || (int64_t) N * W / hop < 1 )
		return fail( ctx, FLAN_B200_INVALID, "need 2 <= window_size <= dft_size and 1 <= hop <= dft_size*window_size" );
	if( !( sr > 0.0f ) || !( ar > 0.0f ) )
		return fail( ctx, FLAN_B200_INVALID, "sample_rate and analysis_rate must be positive" );
	const auto key = std::make_tuple( N, W, hop, fbits( sr ), fbits( ar ) );
	auto it = ctx->plans.find( key );
	if( it != ctx->plans.end() ) { *out = it->second.get(); return FLAN_B200_OK; }
	auto plan = std::make_unique<DevicePlan>();
	if( !build_tables( N, W, hop, sr, ar, plan->host ) )
		return fail( ctx, FLAN_B200_INVALID, "could not build plan tables" );
	cudaError_t e = cudaSuccess;
	auto up = [&]( auto & vec, auto ** d ) { if( e == cudaSuccess ) e = upload_vec( vec, d, ctx->compute ); };
	up( plan->host.win_analysis, &plan->win_analysis ); up( plan->host.win_synthesis, &plan->win_synthesis );
	up( plan->host.expected, &plan->expected ); up( plan->host.binc, &plan->binc );
	up( plan->host.post_tw, &plan->post_tw ); up( plan->host.post_rot, &plan->post_rot );
	up( plan->host.binc4, &plan->binc4 ); up( plan->host.pass_tw, &plan->pass_tw );
	up( plan->host.pass_tw16, &plan->pass_tw16 ); up( plan->host.pass_tw_rev, &plan->pass_tw_rev );
	if( !dft_size_is_templated( N ) )
		{
		// any other size: the run-time-sized transform of pv_generic.cu (power-of-two passes, Bluestein otherwise)
		if( !build_generic( N, plan->generic_host ) ) return fail( ctx, FLAN_B200_INVALID, "could not build the generic transform tables" );
		plan->generic = true;
		up( plan->generic_host.tw, &plan->g_tw ); up( plan->generic_host.chirp, &plan->g_chirp ); up( plan->generic_host.chirp_fft, &plan->g_chirp_fft );
		const GenericHost & h = plan->generic_host;
		plan->generic_fft = GenericFft{ h.N, h.even, h.L, h.B, h.M, h.bluestein, plan->g_tw, plan->g_chirp, plan->g_chirp_fft };
		}
	if( e == cudaSuccess ) e = cudaStreamSynchronize( ctx->compute );     // once per plan: its tables are then visible to every stream
	if( e != cudaSuccess ) { free_plan( plan.get() ); return cuda_fail( ctx, e, "plan upload" ); }
	*out = plan.get();
	ctx->plans[key] = std::move( plan );
	return FLAN_B200_OK;
	}

int get_workspace( flan_b200_ctx * ctx, size_t bytes, void ** out, bool * kept )
	{
	ctx->summaries.drop();          // the caller overwrites them (a producer publishes again after its launch)
	if( kept ) *kept = bytes <= ctx->workspace_bytes;
	if( bytes > ctx->workspace_bytes )
		{
		if( ctx->workspace )
			{
			CK( cudaDeviceSynchronize(), "workspace sync" );
			cudaFree( ctx->workspace );
			ctx->workspace = nullptr; ctx->workspace_bytes = 0;
			}
		bytes = align_up( bytes + bytes / 4, size_t( 1 ) << 20 );       // grow with headroom: sizes creep call by call
		CK( cudaMalloc( &ctx->workspace, bytes ), "workspace alloc" );
		ctx->workspace_bytes = bytes;
		}
	// one scratch area for every stream: a call on another stream than the last user's waits for that user
	if( ctx->ws_recorded && ctx->ws_stream != ctx->compute ) CK( cudaStreamWaitEvent( ctx->compute, ctx->ws_event, 0 ), "workspace wait" );
	ctx->ws_touched = true;
	*out = ctx->workspace;
	return FLAN_B200_OK;
	}

LaunchTimer::LaunchTimer( flan_b200_ctx * c, int k, cudaStream_t on ) : ctx( c ), kind( k ), stream( on ? on : c->compute )
	{
	if( !ctx->timing ) return;
	if( cudaEventCreate( &start ) != cudaSuccess || cudaEventCreate( &stop ) != cudaSuccess ) { start = stop = nullptr; return; }
	cudaEventRecord( start, stream );
	}

LaunchTimer::~LaunchTimer()
	{
	if( kind < 9 ) ctx->launches++;
	if( !start ) return;
	cudaEventRecord( stop, stream );
	ctx->timed.push_back( { kind, start, stop } );
	}

// ---- device blocks and their ordering events --------------------------------------------------------------
Block * find_block( flan_b200_ctx * ctx, const void * p )
	{
	if( !p || ctx->live.empty() ) return nullptr;
	auto it = ctx->live.upper_bound( (uintptr_t) p );
	if( it == ctx->live.begin() ) return nullptr;
	--it;
	Block & b = it->second;
	return ( (uintptr_t) p < (uintptr_t) b.ptr + b.bytes ) ? &b : nullptr;
	}

void main_acquire( flan_b200_ctx * ctx, const void * p )
	{
	Block * b = find_block( ctx, p );
	if( !b ) return;
	if( b->side_pending ) cudaStreamWaitEvent( ctx->compute, b->side_event, 0 );
	if( b->main_pending && b->main_stream != ctx->compute ) cudaStreamWaitEvent( ctx->compute, b->main_event, 0 );
	}

void main_release( flan_b200_ctx * ctx, const void * p )
	{
	Block * b = find_block( ctx, p );
	if( !b ) return;
	cudaEventRecord( b->main_event, ctx->compute );
	b->main_pending = true; b->main_stream = ctx->compute;
	}

// Foreign memory (not from flan_b200_malloc, e.g. a torch tensor): no per-block history, so the copy stream is ordered
// after everything enqueued on the context's stream so far, and the context's stream after the copy.
static cudaEvent_t scratch_event( flan_b200_ctx * ctx )
	{
	static thread_local std::map<flan_b200_ctx *, cudaEvent_t> ev;        // per thread: record + wait pairs never interleave
	cudaEvent_t & e = ev[ctx];
	if( !e ) cudaEventCreateWithFlags( &e, cudaEventDisableTiming );
	return e;
	}

int side_acquire( flan_b200_ctx * ctx, cudaStream_t side, const void * p )
	{
	Block * b = find_block( ctx, p );
	if( b )
		{
		if( b->main_pending ) CK( cudaStreamWaitEvent( side, b->main_event, 0 ), "copy stream wait" );
		if( b->side_pending ) CK( cudaStreamWaitEvent( side, b->side_event, 0 ), "copy stream wait" );
		return FLAN_B200_OK;
		}
	cudaEvent_t e = scratch_event( ctx );
	CK( cudaEventRecord( e, ctx->compute ), "event record" );
	CK( cudaStreamWaitEvent( side, e, 0 ), "copy stream wait" );
	return FLAN_B200_OK;
	}

int side_release( flan_b200_ctx * ctx, cudaStream_t side, const void * p )
	{
	Block * b = find_block( ctx, p );
	if( b )
		{
		CK( cudaEventRecord( b->side_event, side ), "event record" );
		b->side_pending = true;
		return FLAN_B200_OK;
		}
	cudaEvent_t e = scratch_event( ctx );
	CK( cudaEventRecord( e, side ), "event record" );
	CK( cudaStreamWaitEvent( ctx->compute, e, 0 ), "stream wait" );
	return FLAN_B200_OK;
	}

// ---- host staging ----------------------------------------------------------------------------------------------
bool host_is_pinned( const void * p )
	{
	cudaPointerAttributes a{};
	if( cudaPointerGetAttributes( &a, p ) != cudaSuccess ) { cudaGetLastError(); return false; }
	return a.type == cudaMemoryTypeHost;
	}

int ensure_ring( flan_b200_ctx * ctx, PinnedRing & ring )
	{
	if( ring.base ) return FLAN_B200_OK;
	ring.slice = size_t( 4 ) << 20;
	ring.depth = 8;
	CK( cudaMallocHost( (void **) &ring.base, ring.slice * ring.depth ), "pinned staging ring" );
	ring.ev.resize( ring.depth ); ring.armed.assign( ring.depth, 0 );
	for( auto & e : ring.ev ) CK( cudaEventCreateWithFlags( &e, cudaEventDisableTiming ), "event create" );
	return FLAN_B200_OK;
	}

int copy_h2d_2d( flan_b200_ctx * ctx, void * d, size_t d_pitch, const void * h, size_t h_pitch, size_t width, size_t rows )
	{
	if( width == 0 || rows == 0 ) return FLAN_B200_OK;
	if( host_is_pinned( h ) )
		{
		if( rows == 1 || ( d_pitch == width && h_pitch == width ) )
			CK( cudaMemcpyAsync( d, h, width * rows, cudaMemcpyHostToDevice, ctx->h2d ), "upload" );
		else if( rows <= 16 )       // a few channels: plain 1-D DMA per row
			for( size_t r = 0; r < rows; ++r )
				CK( cudaMemcpyAsync( (char *) d + r * d_pitch, (const char *) h + r * h_pitch, width, cudaMemcpyHostToDevice, ctx->h2d ), "upload" );
		else
			CK( cudaMemcpy2DAsync( d, d_pitch, h, h_pitch, width, rows, cudaMemcpyHostToDevice, ctx->h2d ), "upload" );
		return FLAN_B200_OK;
		}
	PinnedRing & ring = ctx->ring_up;
	int rc = ensure_ring( ctx, ring );
	if( rc ) return rc;
	CopyPool & pool = copy_pool( ctx );
	for( size_t r = 0; r < rows; ++r )
		for( size_t off = 0; off < width; off += ring.slice )
			{
			const size_t nb = std::min( ring.slice, width - off );
			const int i = (int)( ring.next++ % ring.depth );
			if( ring.armed[i] ) CK( cudaEventSynchronize( ring.ev[i] ), "staging wait" );
			char * stage = ring.base + ring.slice * i;
			pool.copy( stage, (const char *) h + r * h_pitch + off, nb );
			CK( cudaMemcpyAsync( (char *) d + r * d_pitch + off, stage, nb, cudaMemcpyHostToDevice, ctx->h2d ), "upload" );
			CK( cudaEventRecord( ring.ev[i], ctx->h2d ), "event record" );
			ring.armed[i] = 1;
			}
	return FLAN_B200_OK;
	}

int copy_d2h_2d( flan_b200_ctx * ctx, void * h, size_t h_pitch, const void * d, size_t d_pitch, size_t width, size_t rows )
	{
	if( width == 0 || rows == 0 ) return FLAN_B200_OK;
	if( host_is_pinned( h ) )
		{
		if( rows == 1 || ( d_pitch == width && h_pitch == width ) )
			CK( cudaMemcpyAsync( h, d, width * rows, cudaMemcpyDeviceToHost, ctx->d2h ), "download" );
		else if( rows <= 16 )
			for( size_t r = 0; r < rows; ++r )
				CK( cudaMemcpyAsync( (char *) h + r * h_pitch, (const char *) d + r * d_pitch, width, cudaMemcpyDeviceToHost, ctx->d2h ), "download" );
		else
			CK( cudaMemcpy2DAsync( h, h_pitch, d, d_pitch, width, rows, cudaMemcpyDeviceToHost, ctx->d2h ), "download" );
		return FLAN_B200_OK;
		}
	PinnedRing & ring = ctx->ring_down;
	int rc = ensure_ring( ctx, ring );
	if( rc ) return rc;
	CopyPool & pool = copy_pool( ctx );
	// slices are issued up to `depth` ahead of the one being drained into the pageable destination
	struct Slice { size_t r, off, nb; int i; };
	std::vector<Slice> all;
	for( size_t r = 0; r < rows; ++r )
		for( size_t off = 0; off < width; off += ring.slice )
			all.push_back( { r, off, std::min( ring.slice, width - off ), 0 } );
	size_t issued = 0;
	for( size_t drained = 0; drained < all.size(); ++drained )
		{
		while( issued < all.size() && issued < drained + (size_t) ring.depth )
			{
			Slice & s = all[issued];
			s.i = (int)( ring.next++ % ring.depth );
			CK( cudaMemcpyAsync( ring.base + ring.slice * s.i, (const char *) d + s.r * d_pitch + s.off, s.nb, cudaMemcpyDeviceToHost, ctx->d2h ), "download" );
			CK( cudaEventRecord( ring.ev[s.i], ctx->d2h ), "event record" );
			ring.armed[s.i] = 0;        // drained below before the slot comes round again
			++issued;
			}
		const Slice & s = all[drained];
		CK( cudaEventSynchronize( ring.ev[s.i] ), "staging wait" );
		pool.copy( (char *) h + s.r * h_pitch + s.off, ring.base + ring.slice * s.i, s.nb );
		}
	return FLAN_B200_OK;
	}

// ---- the two transforms over a frame range ---------------------------------------------------------------------

static int seg_len_cap( const flan_b200_ctx * ctx, int N ) { return ctx->max_seg_len ? ctx->max_seg_len : ( N >= 2048 ? 128 : 64 ); }

// 8-byte loads of the input: hop, half window, stride, offset and address all even
static bool audio_aligned2( int W, int hop, const float * audio, int64_t stride, int64_t offset )
	{
	return hop % 2 == 0 && ( W / 2 ) % 2 == 0 && stride % 2 == 0 && offset % 2 == 0 && (uintptr_t) audio % 8 == 0;
	}

// The analysis kernel of a call: the launch policy's choice (pv_policy.h), decided on the whole signal's frame count.
// Development builds apply the overrides of FLAN_B200_PT_ANALYSIS (8, 16 or 17: the mirrored last pass where it fits),
// FLAN_B200_TPS_ANALYSIS and FLAN_B200_ONEBUF here, snapped to the variants they carry.
static TransformKernel analysis_kernel( const flan_b200_ctx * ctx, int N, int W, int hop, int C, int64_t n_total, bool aligned2, bool emit )
	{
	TransformKernel k = choose_analysis( N, W, hop, C, n_total / hop + 1, ctx->sms, aligned2, emit );
#ifdef FLAN_B200_DEBUG
	if( k.kind == KernelKind::generic_analysis ) return k;
	int pt = ctx->pt_analysis ? ctx->pt_analysis : ( k.kind == KernelKind::analysis_mirror ? 17 : k.PT );
	if( pt == 17 && !analysis_mirror_fits( N, W, hop ) ) pt = N >= 4096 ? 16 : 8;
	if( pt != 17 && ( pt != 16 || N < 512 ) ) pt = 8;
	const int tps = ctx->tps_analysis ? ctx->tps_analysis : ( pt == 8 ? 768 : 512 );
	k.kind = pt == 17 ? KernelKind::analysis_mirror : KernelKind::analysis;
	k.PT = pt == 8 ? 8 : 16;
	k.TPS = pt == 8 ? ( tps >= 1024 ? 1024 : tps < 768 ? 512 : 768 ) : ( tps >= 768 ? 768 : tps >= 640 ? 640 : tps < 512 ? 384 : 512 );
	k.ONE = pt != 8 && ctx->one_buffer != 0;
	k.PAD = analysis_pad_fits( k, W, aligned2 );
	k.EMIT = emit && !k.PAD && analysis_emit_fits( k, W );
#endif
	return k;
	}

// The resynthesis kernel: the launch policy's choice. Development builds apply FLAN_B200_SYNTH_VARIANT (17: mirrored
// where it fits, anything else the 8-point kernel), FLAN_B200_TPS_SYNTHESIS and FLAN_B200_SYNTH_ONEBUF.
static TransformKernel synthesis_kernel( const flan_b200_ctx * ctx, int N, int W, int hop )
	{
	TransformKernel k = choose_synthesis( N, W, hop );
#ifdef FLAN_B200_DEBUG
	if( k.kind == KernelKind::generic_synthesis ) return k;
	const bool mirror = ( ctx->synth_variant < 0 || ctx->synth_variant == 17 ) && synthesis_mirror_fits( N, W, hop );
	const bool one = ctx->synth_one_buffer >= 0 ? ctx->synth_one_buffer != 0 : N == 8192;
	const int tps = ctx->tps_synthesis ? ctx->tps_synthesis : ( mirror ? 384 : ( N == 8192 ? 1024 : 768 ) );
	k.kind = mirror ? KernelKind::synthesis_mirror : KernelKind::synthesis;
	k.PT = mirror ? 16 : 8;
	k.GEN = mirror && !standard_shape( N, W, hop );
	if( mirror && N == 8192 ) { k.TPS = one ? 512 : 256; k.ONE = one; }
	else if( mirror && ( tps >= 512 || one ) ) { k.TPS = tps >= 512 ? 512 : 384; k.ONE = one; }
	else if( mirror ) k = choose_synthesis( N, W, hop );
	else if( N == 8192 && tps >= 1024 ) { k.TPS = 1024; k.ONE = true; }
	else { k.TPS = tps >= 1024 ? 1024 : ( tps < 768 ? 512 : 768 ); k.ONE = false; }
#endif
	return k;
	}

// A failed launch or occupancy query of a transform kernel names the kernel. cudaErrorInvalidValue is also what a
// descriptor outside this build's kernel list gives: an internal error of the launch policy.
static int transform_fail( flan_b200_ctx * ctx, cudaError_t e, const TransformKernel & k, const char * what )
	{
	return cuda_fail( ctx, e, ( std::string( e == cudaErrorInvalidValue ? "internal: " : "" ) + what + " of " + k.name() ).c_str() );
	}
#define CK_KERNEL( call, k, what ) do { cudaError_t e_ = ( call ); if( e_ != cudaSuccess ) return transform_fail( ctx, e_, k, what ); } while( 0 )

int analysis_range( flan_b200_ctx * ctx, const AnalysisCall & c )
	{
	const int C = c.C, W = c.W, hop = c.hop, N = c.N;
	if( C < 1 || c.n_total < 0 || hop < 1 )
		return fail( ctx, FLAN_B200_INVALID, "bad channel count, length or hop" );
	const int64_t F = flan_b200_num_frames( c.n_total, hop );
	if( c.frame_begin < 0 || c.frame_end < c.frame_begin || c.frame_end > F )
		return fail( ctx, FLAN_B200_INVALID, "frame range outside [0, n/hop + 1]" );
	DevicePlan * plan = nullptr;
	int rc = get_plan( ctx, N, W, hop, c.sr, flan_b200_analysis_rate( c.sr, hop ), &plan );
	if( rc ) return rc;
	const int64_t frames = c.frame_end - c.frame_begin;
	if( frames == 0 ) return FLAN_B200_OK;
	// the shard must hold every in-signal sample its frames (and the warm-up frame) read
	int64_t need_lo = (int64_t) hop * ( c.frame_begin > 0 ? c.frame_begin - 1 : 0 ) - W / 2;
	int64_t need_hi = (int64_t) hop * ( c.frame_end - 1 ) - W / 2 + W;
	if( need_lo < 0 ) need_lo = 0;
	if( need_hi > c.n_total ) need_hi = c.n_total;
	if( need_hi > need_lo && ( c.audio_offset > need_lo || c.audio_offset + c.audio_len < need_hi ) )
		return fail( ctx, FLAN_B200_INVALID, "local audio does not cover the halo of the requested frame range" );

	int seg_len = choose_seg_len( frames, C, ctx->sms, W, hop, seg_len_cap( ctx, N ), true );
	int segs = (int)( ( frames + seg_len - 1 ) / seg_len );
	AnalysisArgs a{};
	a.audio = c.d_audio_local; a.audio_stride = c.audio_stride; a.audio_offset = c.audio_offset; a.n_total = c.n_total;
	a.pv = (float2 *) c.d_pv_rows; a.pv_channel_stride = c.pv_channel_stride;
	a.frame_begin = c.frame_begin; a.frame_end = c.frame_end;
	a.seg_len = seg_len; a.segs_per_channel = segs;
	a.W = W; a.hop = hop;
	a.aligned2 = audio_aligned2( W, hop, c.d_audio_local, c.audio_stride, c.audio_offset );
	a.win = plan->win_analysis; a.binc = plan->binc; a.binc4 = plan->binc4; a.post_rot = plan->post_rot;
	a.k = plan->host.k;
	if( plan->generic )
		{
		GenericAnalysisArgs ga{};
		ga.a = a; ga.g = plan->generic_fft;
		ga.total_segments = (int64_t) C * segs;
		const GenericGeometry geo = generic_geometry( ga.g, generic_analysis_state_bytes( ga.g ), ga.total_segments, ctx->sms );
		void * ws = nullptr;
		rc = get_workspace( ctx, (size_t)( geo.blocks * geo.scratch_stride ), &ws );
		if( rc ) return rc;
		ga.scratch = (unsigned char *) ws; ga.scratch_stride = geo.scratch_stride; ga.fft_in_smem = geo.fft_in_smem;
		{ LaunchTimer lt( ctx, 0 ); CK( launch_generic_analysis( ga, geo, ctx->compute ), "analysis launch" ); }
		return FLAN_B200_OK;
		}
	// Summaries for a resynthesis of these rows as they are (flan_b200_hint_resynthesis): the kernel that can leave them
	// writes them to the workspace, in the segments resynthesis will use, when the scan that repairs marked entries (three
	// launches) will read them; anything else ignores the hint. (A frame range without emit_seg_len is a shard of a
	// per-GPU process: its resynthesis chooses the segments from the local frame count, and so does this.)
	const int B = N / 2 + 1;
	PhaseLayout lay{};
	if( c.emit_summary && c.pv_channel_stride == frames * (int64_t) B ) lay = phase_layout( ctx, C, frames, B, W, hop, c.emit_seg_len );
	const TransformKernel k = analysis_kernel( ctx, N, W, hop, C, c.n_total, a.aligned2, lay.segs > 256 && lay.seg_len <= 128 );
	a.one_buffer = k.ONE;
	a.pass_tw = k.PT == 16 ? plan->pass_tw16 : plan->pass_tw;
	if( k.EMIT )
		{
		void * ws = nullptr;
		rc = get_workspace( ctx, lay.bytes(), &ws );
		if( rc ) return rc;
		seg_len = lay.seg_len; segs = lay.segs;
		a.seg_len = seg_len; a.segs_per_channel = segs;
		a.seg_out = (PhaseSeg *) ws; a.P = plan->host.P; a.rcpP = plan->host.rcpP;
		CK( cudaMemsetAsync( ctx->summaries.nan_flag, 0, sizeof( int ), ctx->compute ), "flag clear" );
		{ LaunchTimer lt( ctx, 0 ); CK_KERNEL( launch( k, a, (int64_t) C * segs, ctx->compute ), k, "analysis launch" ); }
		ctx->summaries.publish( { c.d_pv_rows, c.pv_channel_stride, c.frame_begin, c.frame_end, C, B, W, seg_len, c.sr, flan_b200_analysis_rate( c.sr, hop ) },
		                        { /* needs_fix */ true, /* nan_known */ true } );
		return FLAN_B200_OK;
		}
	// Whole waves: with a few waves of CTAs the last, partly filled one is a large share of the launch (a 1/8 shard of cfg3:
	// 660 CTAs = 2.23 waves of 296). Segments are shortened until the CTAs just fill the waves they need anyway. Analysis
	// results do not depend on where segments are cut (the warm-up frame recomputes the previous phase exactly).
	if( (int64_t) C * segs > 2 * (int64_t) ctx->sms )
		{
		int per_sm = 0;
		CK_KERNEL( resident_ctas( k, a, &per_sm ), k, "occupancy query" );
		const int64_t wave = (int64_t) ctx->sms * std::max( 1, per_sm );
		const int64_t ctas = (int64_t) C * segs;
		const int64_t per_channel = ( ( ctas + wave - 1 ) / wave * wave ) / C;
		const int64_t shorter = per_channel > 0 ? ( frames + per_channel - 1 ) / per_channel : seg_len;
		if( ctas > wave && shorter >= 8 && shorter < seg_len )
			{
			seg_len = (int) shorter; segs = (int)( ( frames + seg_len - 1 ) / seg_len );
			a.seg_len = seg_len; a.segs_per_channel = segs;
			}
		}
	ctx->summaries.drop();          // new rows, no summaries of them
	{ LaunchTimer lt( ctx, 0 ); CK_KERNEL( launch( k, a, (int64_t) C * segs, ctx->compute ), k, "analysis launch" ); }
	return FLAN_B200_OK;
	}

int64_t ctas_per_slice( int64_t ctas, int64_t wave, size_t copy_bytes )
	{
	if( wave < 1 ) wave = 1;
	const int64_t waves = ( ctas + wave - 1 ) / wave;
	int64_t n = std::min<int64_t>( 8, std::min<int64_t>( waves, (int64_t)( copy_bytes >> 22 ) ) );     // >= 4 MiB of copy per slice
	if( n < 1 ) n = 1;
	return ( ( waves + n - 1 ) / n ) * wave;
	}

int resynthesis_seg_len( const flan_b200_ctx * ctx, int C, int64_t frames, int N, int W, int hop )
	{
	return choose_seg_len( frames, C, ctx->sms, W, hop, seg_len_cap( ctx, N ), false, synth_ctas_per_sm( N ) );
	}

PhaseLayout phase_layout( const flan_b200_ctx * ctx, int C, int64_t frames, int B, int W, int hop, int seg_len_given )
	{
	PhaseLayout l{};
	int seg_len = seg_len_given ? seg_len_given : resynthesis_seg_len( ctx, C, frames, ( B - 1 ) * 2, W, hop );
	if( seg_len > frames ) seg_len = (int) frames;
	if( seg_len < 1 ) seg_len = 1;
	l.seg_len = seg_len;
	l.segs = (int)( ( frames + seg_len - 1 ) / seg_len );
	l.seg_bytes = align_up( sizeof( PhaseSeg ) * (size_t) C * l.segs * B, 256 );
	l.acc_bytes = align_up( sizeof( double ) * (size_t) C * l.segs * B, 256 );
	l.group_len = 32;
	while( ( l.segs + l.group_len - 1 ) / l.group_len > 65535 ) l.group_len *= 2;
	l.groups = ( l.segs + l.group_len - 1 ) / l.group_len;
	l.grp_bytes = align_up( sizeof( PhaseSeg ) * (size_t) C * l.groups * B, 256 );
	return l;
	}

bool PhaseSummaries::Key::operator==( const Key & o ) const
	{
	return pv == o.pv && channel_stride == o.channel_stride && frame_begin == o.frame_begin && frame_end == o.frame_end
	    && C == o.C && B == o.B && W == o.W && seg_len == o.seg_len && fbits( sr ) == fbits( o.sr ) && fbits( ar ) == fbits( o.ar );
	}
void PhaseSummaries::publish( const Key & key, const Source & source ) { key_ = key; source_ = source; valid_ = true; }
std::optional<PhaseSummaries::Source> PhaseSummaries::match( const Key & key, bool need_nan_flag ) const
	{
	if( !valid_ || !( key_ == key ) || ( need_nan_flag && !source_.nan_known ) ) return std::nullopt;
	return source_;
	}
void PhaseSummaries::drop() { valid_ = false; }
void PhaseSummaries::drop_if_within( const Block & b ) { if( (uintptr_t) key_.pv >= (uintptr_t) b.ptr && (uintptr_t) key_.pv < (uintptr_t) b.ptr + b.bytes ) drop(); }

// The promise of flan_b200_promise_unchanged, per calling thread: the next whole-signal resynthesis of exactly this
// buffer may use the phase summaries its producer left in the workspace.
static thread_local const void * g_promised_pv = nullptr;
void promise_unchanged( const void * d_pv ) { g_promised_pv = d_pv; }
// flan_b200_hint_resynthesis, per calling thread: consumed by the next flan_b200_convert_to_pv.
static thread_local bool g_resynthesis_hint = false;
bool take_resynthesis_hint() { const bool h = g_resynthesis_hint; g_resynthesis_hint = false; return h; }
void set_resynthesis_hint() { g_resynthesis_hint = true; }
bool take_promise( const void * d_pv )
	{
	const bool hit = d_pv && g_promised_pv == d_pv;
	g_promised_pv = nullptr;
	return hit;
	}

int synth_range( flan_b200_ctx * ctx, const SynthCall & s )
	{
	const int C = s.C, B = s.B, W = s.W;
	if( C < 1 || B < 2 || s.frame_begin < 0 || s.frame_end < s.frame_begin || s.frames_total < s.frame_end )
		return fail( ctx, FLAN_B200_INVALID, "bad channel / bin / frame-range arguments" );
	const int N = ( B - 1 ) * 2;                                        // PVBuffer.cpp:356-359
	const int hop = flan_b200_hop_from_rates( s.sr, s.ar );
	DevicePlan * plan = nullptr;
	int rc = get_plan( ctx, N, W, hop, s.sr, s.ar, &plan );
	if( rc ) return rc;
	const int64_t frames = s.frame_end - s.frame_begin;
	if( frames == 0 ) return FLAN_B200_OK;
	if( cancelled( s.cancel ) ) return fail( ctx, FLAN_B200_CANCELLED, "cancelled" );

	// s.seg_len: the multi-device forms pass the segment length of the WHOLE signal and cut their shards at multiples of
	// it, so that a shard walks exactly the segments the uncut signal would and gives the same bits
	const PhaseLayout lay = phase_layout( ctx, C, frames, B, W, hop, s.seg_len );
	const int seg_len = lay.seg_len, segs = lay.segs, group_len = lay.group_len, groups = lay.groups;
	const size_t seg_bytes = lay.seg_bytes, acc_bytes = lay.acc_bytes, grp_bytes = lay.grp_bytes;
	// summaries a producer left of exactly these rows, taken before get_workspace drops the record (summaries whose
	// NaN / Inf flag is gone cannot serve a caller that asks for the flag), and forgotten if the workspace had to grow
	const PhaseSummaries::Key key{ s.d_pv_rows, s.pv_channel_stride, s.frame_begin, s.frame_end, C, B, W, seg_len, s.sr, s.ar };
	std::optional<PhaseSummaries::Source> held = s.reuse_summary ? ctx->summaries.match( key, s.d_nan_flag != nullptr ) : std::nullopt;
	GenericSynthArgs ga{};
	GenericGeometry geo{};
	if( plan->generic )       // the per-CTA slabs of the run-time-sized transform go behind the phase scratch
		{
		ga.g = plan->generic_fft;
		geo = generic_geometry( ga.g, generic_synthesis_state_bytes( ga.g, W ), (int64_t) C * segs, ctx->sms );
		}
	const size_t phase_bytes = seg_bytes + acc_bytes + grp_bytes;
	void * ws = nullptr;
	bool kept = false;
	rc = get_workspace( ctx, phase_bytes + (size_t)( geo.blocks * geo.scratch_stride ), &ws, &kept );
	if( rc ) return rc;
	if( !kept ) held.reset();       // a new allocation: what the producer left is gone
	ga.scratch = (unsigned char *) ws + phase_bytes; ga.scratch_stride = geo.scratch_stride; ga.fft_in_smem = geo.fft_in_smem;
	PhaseSeg * d_seg = (PhaseSeg *) ws;
	double * d_acc = (double *)( (char *) ws + seg_bytes );
	PhaseSeg * d_grp = (PhaseSeg *)( (char *) ws + seg_bytes + acc_bytes );

	PhaseSegArgs sa{};
	sa.pv = (const float2 *) s.d_pv_rows; sa.pv_channel_stride = s.pv_channel_stride;
	sa.frame_begin = s.frame_begin; sa.frame_end = s.frame_end;
	sa.seg_len = seg_len; sa.segs_per_channel = segs; sa.B = B;
	sa.seg_out = d_seg; sa.nan_flag = s.d_nan_flag ? s.d_nan_flag : ctx->summaries.sink;
	sa.k = plan->host.k; sa.P = plan->host.P; sa.rcpP = plan->host.rcpP;
	if( !held ) { LaunchTimer lt( ctx, 1 ); CK( launch_phase_seg( sa, C, ctx->compute ), "phase summary launch" ); }

	PhaseScanArgs sc{};
	sc.seg = d_seg; sc.segs_per_channel = segs; sc.B = B;
	sc.group_len = group_len; sc.groups = groups; sc.group = d_grp;
	sc.carry_in = s.d_carry_in; sc.carry_out = s.d_carry_out;
	sc.acc_start = s.summary_only ? nullptr : d_acc;
	sc.P = plan->host.P; sc.rcpP = plan->host.rcpP;
	// A summary-only call without a carry (flan_b200_phase_summary: the shard's own state, before the states of the
	// earlier shards are known) leaves the carry-free group prefixes behind; the range call that follows on the same
	// data then only re-walks the groups, entering each through carry (+) prefix.
	const bool three_launches = segs > 256 || C > 65535;
	sc.expand_only = ( held && held->group_prefix && three_launches && !s.summary_only && !s.d_carry_out ) ? 1 : 0;
	sc.expand_carry = sc.expand_only ? s.d_carry_in : nullptr;
	if( held && held->needs_fix )
		{
		// summaries of the analysis kernel: the group reduction recomputes the entries it marked (the lowest bins, NaN / Inf)
		if( !three_launches || sc.expand_only ) return fail( ctx, FLAN_B200_INVALID, "internal: marked summaries need the three-launch scan" );
		sc.fix_pv = (const float2 *) s.d_pv_rows; sc.fix_channel_stride = s.pv_channel_stride;
		sc.fix_frame_begin = s.frame_begin; sc.fix_frame_end = s.frame_end; sc.fix_seg_len = seg_len;
		sc.fix_k = plan->host.k; sc.fix_nan_flag = ctx->summaries.nan_flag;
		}
	{ LaunchTimer lt( ctx, 2 ); CK( launch_phase_scan( sc, C, ctx->compute ), "phase scan launch" );
	  ctx->launches += three_launches ? ( sc.expand_only ? 0 : ( s.summary_only ? 1 : 2 ) ) : 0; }     // launch_phase_scan: one launch for short signals, else 1 to 3
	if( held && s.d_nan_flag )
		CK( cudaMemcpyAsync( s.d_nan_flag, ctx->summaries.nan_flag, sizeof( int ), cudaMemcpyDeviceToDevice, ctx->compute ), "flag copy" );
	// the summaries stay for the next call on these rows, marked entries repaired by the scan
	ctx->summaries.publish( key, { /* needs_fix */ false, /* nan_known */ held && held->nan_known,
	                               /* group_prefix */ s.summary_only && !s.d_carry_in && three_launches } );
	if( s.summary_only ) return FLAN_B200_OK;
	if( cancelled( s.cancel ) ) return fail( ctx, FLAN_B200_CANCELLED, "cancelled" );

	// The kernels store every sample that only one segment reaches and red.add the rest onto zeros: clear just those
	// (a few per cent of the output) when the frames' windows leave no gaps, everything otherwise.
	if( hop <= W && C < 65535 )
		{ CK( launch_zero_shared( s.d_out, s.out_stride, s.out_offset, s.out_len, C, s.frame_begin, s.frame_end, seg_len, segs, W, hop, ctx->compute ), "output clear" ); ctx->launches++; }
	else
		for( int c = 0; c < C; ++c )
			CK( cudaMemsetAsync( s.d_out + (int64_t) c * s.out_stride, 0, sizeof( float ) * (size_t) s.out_len, ctx->compute ), "output clear" );

	SynthArgs a{};
	a.pv = (const float2 *) s.d_pv_rows; a.pv_channel_stride = s.pv_channel_stride;
	a.frame_begin = s.frame_begin; a.frame_end = s.frame_end;
	a.out = s.d_out; a.out_stride = s.out_stride; a.out_offset = s.out_offset;
	const int64_t total = s.frames_total * hop;                         // AudioPV.cpp:93
	a.out_lo = s.out_offset > 0 ? s.out_offset : 0;
	a.out_hi = ( s.out_offset + s.out_len < total ) ? s.out_offset + s.out_len : total;
	a.acc_start = d_acc;
	a.seg_len = seg_len; a.segs_per_channel = segs;
	a.W = W; a.hop = hop;
	a.aligned2 = ( hop % 2 == 0 ) && ( ( W / 2 ) % 2 == 0 );
	a.win = plan->win_synthesis; a.post_tw = plan->post_tw; a.pass_tw = plan->pass_tw; a.pass_tw_rev = plan->pass_tw_rev;
	a.out_aligned2 = ( s.out_stride % 2 == 0 ) && ( s.out_offset % 2 == 0 ) && ( (uintptr_t) s.d_out % 8 == 0 );
	a.pv_aligned16 = ( (uintptr_t) s.d_pv_rows % 16 == 0 ); a.channels = C;
	a.k = plan->host.k; a.P = plan->host.P; a.rcpP = plan->host.rcpP;
	const TransformKernel kernel = synthesis_kernel( ctx, N, W, hop );
	a.one_buffer = kernel.ONE;
	// One launch, or -- for the pipelined host forms -- slices of whole waves of CTAs so that a download can follow each.
	int segs_per_slice = segs;
	if( s.on_chunk && s.head_segments <= 0 )
		{
		int64_t wave = ctx->sms;
		if( plan->generic ) wave = geo.blocks;
		else
			{
			int per_sm = 0;
			CK_KERNEL( resident_ctas( kernel, a, &per_sm ), kernel, "occupancy query" );
			wave = (int64_t) ctx->sms * std::max( 1, per_sm );
			}
		segs_per_slice = (int) std::max<int64_t>( 1, ctas_per_slice( (int64_t) C * segs, wave, s.copy_bytes ) / C );
		}
	auto launch_segments = [&]( int s0, int s1, cudaStream_t st, bool timed ) -> int
		{
		a.seg_first = s0; a.seg_count = s1 - s0;
		std::unique_ptr<LaunchTimer> lt;
		if( timed ) lt.reset( new LaunchTimer( ctx, 3 ) ); else ctx->launches++;
		if( plan->generic ) { ga.a = a; CK( launch_generic_synthesis( ga, geo, st ), "synthesis launch" ); }
		else CK_KERNEL( launch( kernel, a, (int64_t) C * ( s1 - s0 ), st ), kernel, "synthesis launch" );
		return FLAN_B200_OK;
		};
	if( s.head_segments > 0 && !plan->generic )
		{
		// the head of the shard beside its interior (the generic kernels share per-CTA slabs of scratch between launches:
		// they take the sliced form below)
		const int sh = std::min( segs, s.head_segments );
		CK( cudaEventRecord( ctx->head_fork, ctx->compute ), "event record" );
		CK( cudaStreamWaitEvent( ctx->s_head, ctx->head_fork, 0 ), "stream wait" );
		rc = launch_segments( 0, sh, ctx->s_head, false );
		if( rc ) return rc;
		if( s.head_event ) CK( cudaEventRecord( s.head_event, ctx->s_head ), "event record" );
		CK( cudaEventRecord( ctx->head_join, ctx->s_head ), "event record" );
		if( sh < segs ) { rc = launch_segments( sh, segs, ctx->compute, true ); if( rc ) return rc; }
		CK( cudaStreamWaitEvent( ctx->compute, ctx->head_join, 0 ), "stream wait" );
		return FLAN_B200_OK;
		}
	int k = 0;
	for( int s0 = 0; s0 < segs; ++k )
		{
		int s1 = std::min( segs, s0 + segs_per_slice );
		if( s.head_segments > 0 ) s1 = ( s0 == 0 ) ? std::min( segs, s.head_segments ) : segs;
		rc = launch_segments( s0, s1, ctx->compute, true );
		if( rc ) return rc;
		if( s.head_segments > 0 && k == 0 && s.head_event ) CK( cudaEventRecord( s.head_event, ctx->compute ), "event record" );
		if( s.on_chunk )
			{
			// frames from segment s1 on touch samples >= hop * fa(s1) - W/2: everything below is final
			int64_t done = ( s1 >= segs ) ? a.out_hi : (int64_t) hop * ( s.frame_begin + (int64_t) s1 * seg_len ) - W / 2;
			if( done < a.out_lo ) done = a.out_lo;
			if( done > a.out_hi ) done = a.out_hi;
			rc = s.on_chunk( k, done );
			if( rc ) return rc;
			}
		s0 = s1;
		}
	return FLAN_B200_OK;
	}

} // namespace pvrt

// ------------------------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------------------------
namespace {

thread_local std::string g_create_error;

int new_block( flan_b200_ctx * ctx, size_t bytes, Block & b )
	{
	cudaError_t e = cudaMalloc( &b.ptr, bytes );
	if( e == cudaErrorMemoryAllocation && !ctx->cached.empty() )
		{
		// give the cached blocks back to the driver and try once more
		cudaGetLastError();
		cudaDeviceSynchronize();
		for( auto & kv : ctx->cached ) { cudaFree( kv.second.ptr ); cudaEventDestroy( kv.second.main_event ); cudaEventDestroy( kv.second.side_event ); }
		ctx->cached.clear(); ctx->cached_bytes = 0;
		e = cudaMalloc( &b.ptr, bytes );
		}
	if( e != cudaSuccess ) { cudaGetLastError(); return cuda_fail( ctx, e, "device alloc" ); }
	b.bytes = bytes;
	CK( cudaEventCreateWithFlags( &b.main_event, cudaEventDisableTiming ), "event create" );
	CK( cudaEventCreateWithFlags( &b.side_event, cudaEventDisableTiming ), "event create" );
	return FLAN_B200_OK;
	}

} // namespace

extern "C" {

int flan_b200_device_count( void )
	{
	int n = 0;
	if( cudaGetDeviceCount( &n ) != cudaSuccess ) return 0;
	return n;
	}

int flan_b200_create( int device, flan_b200_ctx ** out )
	{
	if( !out ) return FLAN_B200_INVALID;
	*out = nullptr;
	int n = 0;
	cudaError_t e = cudaGetDeviceCount( &n );
	if( e != cudaSuccess || n < 1 )
		{
		g_create_error = std::string( "no CUDA device: " ) + ( e != cudaSuccess ? cudaGetErrorString( e ) : "device count is 0" )
		               + " (flan_b200 has no CPU fallback)";
		return FLAN_B200_CUDA;
		}
	if( device < 0 || device >= n ) { g_create_error = "device index out of range"; return FLAN_B200_INVALID; }
	e = cudaSetDevice( device );
	if( e != cudaSuccess ) { g_create_error = cudaGetErrorString( e ); return FLAN_B200_CUDA; }
	cudaDeviceProp prop;
	e = cudaGetDeviceProperties( &prop, device );
	if( e != cudaSuccess ) { g_create_error = cudaGetErrorString( e ); return FLAN_B200_CUDA; }
	if( prop.major < 10 )
		{
		g_create_error = "flan_b200 kernels are built for sm_100a only; device is sm_" + std::to_string( prop.major * 10 + prop.minor );
		return FLAN_B200_CUDA;
		}
	auto * ctx = new flan_b200_ctx;
	ctx->device = device;
#ifdef FLAN_B200_DEBUG
	if( const char * v = std::getenv( "FLAN_B200_TPS_ANALYSIS" ) ) ctx->tps_analysis = std::atoi( v );
	if( const char * v = std::getenv( "FLAN_B200_TPS_SYNTHESIS" ) ) ctx->tps_synthesis = std::atoi( v );
	if( const char * v = std::getenv( "FLAN_B200_PT_ANALYSIS" ) ) ctx->pt_analysis = std::atoi( v );
	if( const char * v = std::getenv( "FLAN_B200_ONEBUF" ) ) ctx->one_buffer = std::atoi( v );
	if( const char * v = std::getenv( "FLAN_B200_SYNTH_ONEBUF" ) ) ctx->synth_one_buffer = std::atoi( v );
	if( const char * v = std::getenv( "FLAN_B200_SEG_LEN" ) ) { const int x = std::atoi( v ); if( x >= 4 ) ctx->max_seg_len = x; }
	if( const char * v = std::getenv( "FLAN_B200_SYNTH_VARIANT" ) ) ctx->synth_variant = std::atoi( v );
#endif
	ctx->sms = prop.multiProcessorCount;
	e = cudaMalloc( (void **) &ctx->d_flags, sizeof( int ) * ( flan_b200_ctx::FLAG_SLOTS + 2 ) );
	if( e == cudaSuccess ) e = cudaMemset( ctx->d_flags, 0, sizeof( int ) * ( flan_b200_ctx::FLAG_SLOTS + 2 ) );
	if( e == cudaSuccess ) e = cudaMallocHost( (void **) &ctx->h_flags, sizeof( int ) * flan_b200_ctx::FLAG_SLOTS );
	if( e == cudaSuccess ) std::memset( ctx->h_flags, 0, sizeof( int ) * flan_b200_ctx::FLAG_SLOTS );
	if( e == cudaSuccess ) e = cudaMalloc( (void **) &ctx->d_check, sizeof( pvm::MapCheck ) );
	if( e == cudaSuccess ) e = cudaStreamCreateWithFlags( &ctx->h2d, cudaStreamNonBlocking );
	if( e == cudaSuccess ) e = cudaStreamCreateWithFlags( &ctx->d2h, cudaStreamNonBlocking );
	if( e == cudaSuccess ) e = cudaStreamCreateWithFlags( &ctx->s_ana, cudaStreamNonBlocking );
	if( e == cudaSuccess ) e = cudaStreamCreateWithFlags( &ctx->s_syn, cudaStreamNonBlocking );
	if( e == cudaSuccess ) e = cudaEventCreateWithFlags( &ctx->ws_event, cudaEventDisableTiming );
		{
		int lo = 0, hi = 0;                                             // numerically lower = higher priority
		if( e == cudaSuccess ) e = cudaDeviceGetStreamPriorityRange( &lo, &hi );
		if( e == cudaSuccess ) e = cudaStreamCreateWithPriority( &ctx->s_head, cudaStreamNonBlocking, hi );
		}
	if( e == cudaSuccess ) e = cudaEventCreateWithFlags( &ctx->head_fork, cudaEventDisableTiming );
	if( e == cudaSuccess ) e = cudaEventCreateWithFlags( &ctx->head_join, cudaEventDisableTiming );
	if( e != cudaSuccess ) { g_create_error = cudaGetErrorString( e ); flan_b200_destroy( ctx ); return FLAN_B200_CUDA; }
	ctx->summaries.sink = ctx->d_flags + flan_b200_ctx::FLAG_SLOTS;
	ctx->summaries.nan_flag = ctx->d_flags + flan_b200_ctx::FLAG_SLOTS + 1;
	*out = ctx;
	return FLAN_B200_OK;
	}

void flan_b200_destroy( flan_b200_ctx * ctx )
	{
	if( !ctx ) return;
	cudaSetDevice( ctx->device );
	cudaStreamSynchronize( ctx->stream );
	for( cudaStream_t * st : { &ctx->s_ana, &ctx->s_syn, &ctx->s_head } ) if( *st ) { cudaStreamSynchronize( *st ); cudaStreamDestroy( *st ); }
	for( cudaEvent_t ev : { ctx->ws_event, ctx->head_fork, ctx->head_join } ) if( ev ) cudaEventDestroy( ev );
	if( ctx->h2d ) { cudaStreamSynchronize( ctx->h2d ); cudaStreamDestroy( ctx->h2d ); }
	if( ctx->d2h ) { cudaStreamSynchronize( ctx->d2h ); cudaStreamDestroy( ctx->d2h ); }
	for( auto & kv : ctx->plans ) free_plan( kv.second.get() );
	for( auto & t : ctx->timed ) { cudaEventDestroy( t.start ); cudaEventDestroy( t.stop ); }
	for( auto * m : { &ctx->live } )
		for( auto & kv : *m ) { cudaFree( kv.second.ptr ); cudaEventDestroy( kv.second.main_event ); cudaEventDestroy( kv.second.side_event ); }
	for( auto & kv : ctx->cached ) { cudaFree( kv.second.ptr ); cudaEventDestroy( kv.second.main_event ); cudaEventDestroy( kv.second.side_event ); }
	for( PinnedRing * r : { &ctx->ring_up, &ctx->ring_down } )
		{
		for( auto & e : r->ev ) cudaEventDestroy( e );
		if( r->base ) cudaFreeHost( r->base );
		}
	if( ctx->workspace ) cudaFree( ctx->workspace );
	cudaFree( ctx->d_flags );
	if( ctx->h_flags ) cudaFreeHost( ctx->h_flags );
	cudaFree( ctx->d_check );
	delete ctx;
	}

const char * flan_b200_last_error( const flan_b200_ctx * ctx )
	{
	return ctx ? thread_error().c_str() : g_create_error.c_str();
	}

int flan_b200_set_stream( flan_b200_ctx * ctx, void * cuda_stream )
	{
	if( !ctx ) return FLAN_B200_INVALID;
	CallLock lock( ctx );
	ctx->stream = (cudaStream_t) cuda_stream;
	ctx->compute = ctx->stream;
	return FLAN_B200_OK;
	}

int flan_b200_synchronize( flan_b200_ctx * ctx )
	{
	if( !ctx ) return FLAN_B200_INVALID;
	cudaStream_t st[5];
		{ CallLock lock( ctx ); st[0] = ctx->stream; st[1] = ctx->h2d; st[2] = ctx->d2h; st[3] = ctx->s_ana; st[4] = ctx->s_syn; }
	// outside the lock: other threads keep enqueueing while this one waits
	for( cudaStream_t s : st ) CK( cudaStreamSynchronize( s ), "synchronize" );
	return FLAN_B200_OK;
	}

static int wait_block( flan_b200_ctx * ctx, const void * d_ptr, bool kernels_too )
	{
	if( !ctx ) return FLAN_B200_INVALID;
	cudaEvent_t side = nullptr, main = nullptr;
		{
		CallLock lock( ctx );
		if( Block * b = find_block( ctx, d_ptr ) )
			{
			if( b->side_pending ) side = b->side_event;
			if( b->main_pending && kernels_too ) main = b->main_event;
			}
		else return flan_b200_synchronize( ctx );
		}
	// outside the lock: other threads keep enqueueing while this one waits (blocks are cached, so the events outlive the wait)
	if( main ) CK( cudaEventSynchronize( main ), "wait" );
	if( side ) CK( cudaEventSynchronize( side ), "wait" );
	return FLAN_B200_OK;
	}

int flan_b200_wait( flan_b200_ctx * ctx, const void * d_ptr ) { return wait_block( ctx, d_ptr, true ); }
int flan_b200_wait_copies( flan_b200_ctx * ctx, const void * d_ptr ) { return wait_block( ctx, d_ptr, false ); }

int flan_b200_sm_count( const flan_b200_ctx * ctx ) { return ctx ? ctx->sms : 0; }
int64_t flan_b200_launch_count( const flan_b200_ctx * ctx ) { return ctx ? ctx->launches : 0; }

int flan_b200_set_timing( flan_b200_ctx * ctx, int enabled )
	{
	if( !ctx ) return FLAN_B200_INVALID;
	CallLock lock( ctx );
	ctx->timing = enabled != 0;
	return FLAN_B200_OK;
	}

int flan_b200_kernel_time( flan_b200_ctx * ctx, int kind, double * total_ms, int64_t * launches )
	{
	if( !ctx || !total_ms || !launches ) return FLAN_B200_INVALID;
	CallLock lock( ctx );
	for( cudaStream_t st : { ctx->stream, ctx->s_ana, ctx->s_syn } ) CK( cudaStreamSynchronize( st ), "timing sync" );
	double ms = 0.0; int64_t n = 0;
	std::vector<flan_b200_ctx::Timed> keep;
	for( auto & t : ctx->timed )
		{
		if( t.kind != kind ) { keep.push_back( t ); continue; }
		float f = 0.0f;
		if( cudaEventElapsedTime( &f, t.start, t.stop ) == cudaSuccess ) { ms += f; ++n; }
		cudaEventDestroy( t.start ); cudaEventDestroy( t.stop );
		}
	ctx->timed.swap( keep );
	*total_ms = ms; *launches = n;
	return FLAN_B200_OK;
	}

// Timeline of everything timed since flan_b200_set_timing( 1 ): (kind, start ms, stop ms) relative to the first entry;
// kinds as flan_b200_kernel_time, plus 9 = upload slice, 10 = download slice of the pipelined host forms. Synchronises
// the device; the entries are consumed.
int flan_b200_trace( flan_b200_ctx * ctx, int * kinds, double * start_ms, double * stop_ms, int capacity, int * count )
	{
	if( !ctx || !count ) return FLAN_B200_INVALID;
	CallLock lock( ctx );
	CK( cudaDeviceSynchronize(), "trace sync" );
	int n = 0;
	cudaEvent_t base = ctx->timed.empty() ? nullptr : ctx->timed.front().start;
	for( auto & t : ctx->timed )
		{
		float a = 0.0f, b = 0.0f;
		if( n < capacity && cudaEventElapsedTime( &a, base, t.start ) == cudaSuccess && cudaEventElapsedTime( &b, base, t.stop ) == cudaSuccess )
			{ kinds[n] = t.kind; start_ms[n] = a; stop_ms[n] = b; ++n; }
		}
	for( auto & t : ctx->timed ) { cudaEventDestroy( t.start ); cudaEventDestroy( t.stop ); }
	ctx->timed.clear();
	*count = n;
	return FLAN_B200_OK;
	}

int flan_b200_malloc( flan_b200_ctx * ctx, size_t bytes, void ** d_out )
	{
	if( !ctx || !d_out ) return FLAN_B200_INVALID;
	CallLock lock( ctx );
	bytes = align_up( bytes ? bytes : 1, 512 );
	Block b;
	auto it = ctx->cached.lower_bound( bytes );
	if( it != ctx->cached.end() && it->first <= bytes + std::max( bytes / 8, size_t( 1 ) << 20 ) )
		{
		b = it->second;
		ctx->cached_bytes -= b.bytes;
		ctx->cached.erase( it );
		}
	else
		{
		int rc = new_block( ctx, bytes, b );
		if( rc ) return rc;
		}
	ctx->live[(uintptr_t) b.ptr] = b;
	*d_out = b.ptr;
	return FLAN_B200_OK;
	}

int flan_b200_free( flan_b200_ctx * ctx, void * d_ptr )
	{
	if( !ctx ) return FLAN_B200_INVALID;
	if( !d_ptr ) return FLAN_B200_OK;
	CallLock lock( ctx );
	auto it = ctx->live.find( (uintptr_t) d_ptr );
	if( it == ctx->live.end() )
		{
		CK( cudaFree( d_ptr ), "device free" );        // not one of ours
		return FLAN_B200_OK;
		}
	Block b = it->second;
	ctx->live.erase( it );
	// the next owner orders itself after the block's last use (its event), or -- for a block no entry point has
	// touched -- after everything enqueued on the stream up to here; copies in flight are covered by side_event
	if( !b.main_pending ) { cudaEventRecord( b.main_event, ctx->stream ); b.main_pending = true; b.main_stream = ctx->stream; }
	ctx->cached.emplace( b.bytes, b );
	ctx->cached_bytes += b.bytes;
	ctx->summaries.drop_if_within( b );
	return FLAN_B200_OK;
	}

int flan_b200_trim( flan_b200_ctx * ctx )
	{
	if( !ctx ) return FLAN_B200_INVALID;
	CallLock lock( ctx );
	CK( cudaDeviceSynchronize(), "trim sync" );
	for( auto & kv : ctx->cached ) { cudaFree( kv.second.ptr ); cudaEventDestroy( kv.second.main_event ); cudaEventDestroy( kv.second.side_event ); }
	ctx->cached.clear(); ctx->cached_bytes = 0;
	return FLAN_B200_OK;
	}

int flan_b200_upload( flan_b200_ctx * ctx, void * d_dst, const void * h_src, size_t bytes )
	{
	if( !ctx ) return FLAN_B200_INVALID;
	if( bytes == 0 ) return FLAN_B200_OK;
	CallLock lock( ctx );
	int rc = side_acquire( ctx, ctx->h2d, d_dst );
	if( !rc ) rc = copy_h2d_2d( ctx, d_dst, bytes, h_src, bytes, bytes, 1 );
	if( !rc ) rc = side_release( ctx, ctx->h2d, d_dst );
	return rc;
	}

int flan_b200_download( flan_b200_ctx * ctx, void * h_dst, const void * d_src, size_t bytes )
	{
	if( !ctx ) return FLAN_B200_INVALID;
	if( bytes == 0 ) return FLAN_B200_OK;
	CallLock lock( ctx );
	int rc = side_acquire( ctx, ctx->d2h, d_src );
	if( !rc ) rc = copy_d2h_2d( ctx, h_dst, bytes, d_src, bytes, bytes, 1 );
	if( !rc ) rc = side_release( ctx, ctx->d2h, d_src );
	return rc;
	}

int flan_b200_host_register( flan_b200_ctx * ctx, void * h_ptr, size_t bytes )
	{
	if( !ctx || !h_ptr ) return FLAN_B200_INVALID;
	cudaSetDevice( ctx->device );
	CK( cudaHostRegister( h_ptr, bytes, cudaHostRegisterPortable ), "host register" );
	return FLAN_B200_OK;
	}

int flan_b200_host_unregister( flan_b200_ctx * ctx, void * h_ptr )
	{
	if( !ctx || !h_ptr ) return FLAN_B200_INVALID;
	cudaSetDevice( ctx->device );
	CK( cudaHostUnregister( h_ptr ), "host unregister" );
	return FLAN_B200_OK;
	}

int64_t flan_b200_num_frames( int64_t n, int hop )
	{
	if( hop < 1 ) return 0;
	return n / hop + 1;                                 // AudioPV.cpp:17
	}

int flan_b200_hop_from_rates( float sample_rate, float analysis_rate )
	{
	return (int)( sample_rate / analysis_rate );        // PVBuffer.cpp:381-384
	}

float flan_b200_analysis_rate( float sample_rate, int hop )
	{
	return sample_rate / hop;                           // AudioPV.cpp:25
	}

int flan_b200_convert_to_pv_range( flan_b200_ctx * ctx, const float * d_audio_local, int64_t audio_stride,
                                   int64_t audio_offset, int64_t audio_len, int C, int64_t n_total,
                                   float sr, int W, int hop, int N,
                                   int64_t frame_begin, int64_t frame_end,
                                   float * d_pv_rows, int64_t pv_channel_stride )
	{
	if( !ctx ) return FLAN_B200_INVALID;
	CallLock lock( ctx );
	BlockUse use( ctx, { d_audio_local, d_pv_rows } );
	AnalysisCall a{ d_audio_local, audio_stride, audio_offset, audio_len, C, n_total, sr, W, hop, N, frame_begin, frame_end, d_pv_rows, pv_channel_stride };
	a.emit_summary = take_resynthesis_hint();
	return analysis_range( ctx, a );
	}

int flan_b200_convert_to_pv( flan_b200_ctx * ctx, const float * d_audio, int C, int64_t n,
                             float sr, int W, int hop, int N, float * d_pv, const volatile int * cancel )
	{
	if( !ctx ) return FLAN_B200_INVALID;
	if( cancelled( cancel ) ) return fail( ctx, FLAN_B200_CANCELLED, "cancelled" );
	if( hop < 1 ) return fail( ctx, FLAN_B200_INVALID, "hop must be >= 1" );
	const int64_t F = flan_b200_num_frames( n, hop );
	int rc;
		{
		CallLock lock( ctx );
		BlockUse use( ctx, { d_audio, d_pv } );
		AnalysisCall a{ d_audio, n, 0, n, C, n, sr, W, hop, N, 0, F, d_pv, F * ( N / 2 + 1 ) };
		a.emit_summary = take_resynthesis_hint();
		rc = analysis_range( ctx, a );
		}
	if( rc ) return rc;
	if( cancelled( cancel ) ) return fail( ctx, FLAN_B200_CANCELLED, "cancelled" );
	return FLAN_B200_OK;
	}

int flan_b200_convert_to_audio( flan_b200_ctx * ctx, const float * d_pv, int C, int64_t F, int B,
                                float sr, float ar, int W, float * d_audio_out,
                                const volatile int * cancel, int * nan_or_inf )
	{
	if( !ctx ) return FLAN_B200_INVALID;
	if( !( ar > 0.0f ) || !( sr > 0.0f ) ) return fail( ctx, FLAN_B200_INVALID, "rates must be positive" );
	const int hop = flan_b200_hop_from_rates( sr, ar );
	if( hop < 1 ) return fail( ctx, FLAN_B200_INVALID, "analysis_rate above sample_rate gives hop 0" );
	const int64_t out_n = F * hop;
	cudaStream_t st;
		{
		CallLock lock( ctx );
		BlockUse use( ctx, { d_pv, d_audio_out } );
		st = ctx->compute;
		SynthCall s{ d_pv, F * B, C, 0, F, F, B, sr, ar, W };
		s.d_out = d_audio_out; s.out_stride = out_n; s.out_offset = 0; s.out_len = out_n; s.cancel = cancel;
		s.reuse_summary = take_promise( d_pv );
		int * d_flag = nullptr;
		if( nan_or_inf )
			{
			d_flag = ctx->d_flags + ( ctx->flag_next++ % flan_b200_ctx::FLAG_SLOTS );
			CK( cudaMemsetAsync( d_flag, 0, sizeof( int ), st ), "flag clear" );
			s.d_nan_flag = d_flag;
			}
		int rc = synth_range( ctx, s );
		if( rc ) return rc;
		if( nan_or_inf ) CK( cudaMemcpyAsync( nan_or_inf, d_flag, sizeof( int ), cudaMemcpyDeviceToHost, st ), "flag read" );
		}
	if( nan_or_inf ) CK( cudaStreamSynchronize( st ), "flag sync" );
	if( cancelled( cancel ) ) return fail( ctx, FLAN_B200_CANCELLED, "cancelled" );
	return FLAN_B200_OK;
	}

int flan_b200_hint_resynthesis( flan_b200_ctx * ctx )
	{
	if( !ctx ) return FLAN_B200_INVALID;
	pvrt::set_resynthesis_hint();
	return FLAN_B200_OK;
	}

int flan_b200_promise_unchanged( flan_b200_ctx * ctx, const float * d_pv )
	{
	if( !ctx ) return FLAN_B200_INVALID;
	promise_unchanged( d_pv );
	return FLAN_B200_OK;
	}

int flan_b200_phase_summary( flan_b200_ctx * ctx, const float * d_pv_rows, int64_t pv_channel_stride,
                             int C, int64_t frame_begin, int64_t frame_end, int B,
                             float sr, float ar, int W, flan_b200_phase_state * d_state_out )
	{
	if( !ctx || !d_state_out ) return FLAN_B200_INVALID;
	CallLock lock( ctx );
	BlockUse use( ctx, { d_pv_rows, d_state_out } );
	if( frame_end == frame_begin )
		{
		CK( cudaMemsetAsync( d_state_out, 0, sizeof( PhaseSeg ) * (size_t) C * B, ctx->compute ), "state clear" );
		return FLAN_B200_OK;
		}
	SynthCall s{ d_pv_rows, pv_channel_stride, C, frame_begin, frame_end, frame_end, B, sr, ar, W };
	s.d_carry_out = (PhaseSeg *) d_state_out; s.summary_only = true;
	s.reuse_summary = take_promise( d_pv_rows );      // summaries the shard's analysis left (flan_b200_hint_resynthesis)
	return synth_range( ctx, s );
	}

int flan_b200_phase_carry( flan_b200_ctx * ctx, const flan_b200_phase_state * d_all, int rank,
                           int C, int B, flan_b200_phase_state * d_carry_out )
	{
	if( !ctx || rank < 0 || C < 1 || B < 1 ) return FLAN_B200_INVALID;
	CallLock lock( ctx );
	BlockUse use( ctx, { d_all, d_carry_out } );
	const double P = (double)( std::acos( -1.0f ) * 2.0f );
	{ LaunchTimer lt( ctx, 4 ); CK( launch_phase_carry( (const PhaseSeg *) d_all, rank, (int64_t) C * B, (PhaseSeg *) d_carry_out, P, 1.0 / P, ctx->compute ), "phase carry launch" ); }
	return FLAN_B200_OK;
	}

int flan_b200_convert_to_audio_range( flan_b200_ctx * ctx, const float * d_pv_rows, int64_t pv_channel_stride,
                                      int C, int64_t frame_begin, int64_t frame_end, int64_t frames_total,
                                      int B, float sr, float ar, int W,
                                      const flan_b200_phase_state * d_carry_in, int reuse_summary,
                                      float * d_out_local, int64_t out_stride, int64_t out_offset, int64_t out_len )
	{
	return flan_b200_convert_to_audio_range_head( ctx, d_pv_rows, pv_channel_stride, C, frame_begin, frame_end, frames_total, B, sr, ar, W,
	                                              d_carry_in, reuse_summary, d_out_local, out_stride, out_offset, out_len, nullptr );
	}

// The same, with the frames whose windows reach into the previous shard launched FIRST when `head_event` (a cudaEvent_t of
// the caller) is given: it is recorded on the stream right after them, so the caller can send the window - hop partial sums
// at the head of d_out_local to the previous rank on another stream while the rest of the frames compute.
int flan_b200_convert_to_audio_range_head( flan_b200_ctx * ctx, const float * d_pv_rows, int64_t pv_channel_stride,
                                           int C, int64_t frame_begin, int64_t frame_end, int64_t frames_total,
                                           int B, float sr, float ar, int W,
                                           const flan_b200_phase_state * d_carry_in, int reuse_summary,
                                           float * d_out_local, int64_t out_stride, int64_t out_offset, int64_t out_len,
                                           void * head_event )
	{
	if( !ctx ) return FLAN_B200_INVALID;
	if( !( ar > 0.0f ) || !( sr > 0.0f ) || flan_b200_hop_from_rates( sr, ar ) < 1 )
		return fail( ctx, FLAN_B200_INVALID, "bad rates" );
	CallLock lock( ctx );
	BlockUse use( ctx, { d_pv_rows, d_carry_in, d_out_local } );
	SynthCall s{ d_pv_rows, pv_channel_stride, C, frame_begin, frame_end, frames_total, B, sr, ar, W };
	s.d_carry_in = (const PhaseSeg *) d_carry_in; s.reuse_summary = reuse_summary != 0;
	s.d_out = d_out_local; s.out_stride = out_stride; s.out_offset = out_offset; s.out_len = out_len;
	if( head_event )
		{
		// the first segment holds every frame that reaches the previous shard (a segment is at least window / hop frames)
		s.head_segments = 1;
		s.head_event = (cudaEvent_t) head_event;
		}
	return synth_range( ctx, s );
	}

int flan_b200_add( flan_b200_ctx * ctx, float * d_out, const float * d_add, int64_t n )
	{
	if( !ctx ) return FLAN_B200_INVALID;
	if( n <= 0 ) return FLAN_B200_OK;
	CallLock lock( ctx );
	BlockUse use( ctx, { d_out, d_add } );
	{ LaunchTimer lt( ctx, 4 ); CK( launch_add( d_out, d_add, n, ctx->sms, ctx->compute ), "add launch" ); }
	return FLAN_B200_OK;
	}

int flan_b200_mid_side( flan_b200_ctx * ctx, const float * d_in, float * d_out, int64_t n )
	{
	if( !ctx ) return FLAN_B200_INVALID;
	if( n <= 0 ) return FLAN_B200_OK;
	CallLock lock( ctx );
	BlockUse use( ctx, { d_in, d_out } );
	{ LaunchTimer lt( ctx, 4 ); CK( launch_mid_side( d_in, d_out, n, ctx->sms, ctx->compute ), "mid/side launch" ); }
	return FLAN_B200_OK;
	}

// ---- pipelined host-buffer forms ---------------------------------------------------------------------------------

int flan_b200_convert_to_pv_h2d( flan_b200_ctx * ctx, const float * h_audio, float * d_audio, int C, int64_t n,
                                 float sr, int W, int hop, int N, float * d_pv, const volatile int * cancel )
	{
	if( !ctx || !h_audio || !d_audio || !d_pv ) return FLAN_B200_INVALID;
	if( cancelled( cancel ) ) return fail( ctx, FLAN_B200_CANCELLED, "cancelled" );
	if( hop < 1 || C < 1 || n < 0 || W < 2 ) return fail( ctx, FLAN_B200_INVALID, "bad shape" );
	CallLock lock( ctx );
	// library blocks carry their own ordering: the call runs on the analysis stream, beside other callers' kernels
	if( find_block( ctx, d_audio ) && find_block( ctx, d_pv ) ) ctx->compute = ctx->s_ana;
	const int64_t F = flan_b200_num_frames( n, hop );
	const int B = N / 2 + 1;
	DevicePlan * plan = nullptr;
	int rc = get_plan( ctx, N, W, hop, sr, flan_b200_analysis_rate( sr, hop ), &plan );     // argument errors before any copy
	if( rc ) return rc;
	// slices of whole waves of the analysis kernel's CTAs (a partial wave at the end of every slice would be paid each time)
	const int cap = seg_len_cap( ctx, N );
	int64_t wave = ctx->sms;
	if( plan->generic )
		{
		const int seg_len = choose_seg_len( F, C, ctx->sms, W, hop, cap, true );
		wave = generic_geometry( plan->generic_fft, generic_analysis_state_bytes( plan->generic_fft ), ( F + seg_len - 1 ) / seg_len * C, ctx->sms ).blocks;
		}
	else
		{
		const TransformKernel k = analysis_kernel( ctx, N, W, hop, C, n, audio_aligned2( W, hop, d_audio, n, 0 ), false );
		AnalysisArgs q{};
		q.one_buffer = k.ONE;
		int per_sm = 0;
		CK_KERNEL( resident_ctas( k, q, &per_sm ), k, "occupancy query" );
		wave = (int64_t) ctx->sms * std::max( 1, per_sm );
		}
	const int64_t ctas = ( F + cap - 1 ) / cap * C;
	const int64_t frames_per_slice = std::max<int64_t>( 1, ctas_per_slice( ctas, wave, sizeof( float ) * (size_t) C * n ) / C ) * cap;
	const int slices = (int)( ( F + frames_per_slice - 1 ) / frames_per_slice );
	rc = side_acquire( ctx, ctx->h2d, d_audio );
	if( rc ) return rc;
	main_acquire( ctx, d_pv );
	std::vector<cudaEvent_t> & ev = ctx->slice_events;
	while( (int) ev.size() < slices ) { cudaEvent_t e; CK( cudaEventCreateWithFlags( &e, cudaEventDisableTiming ), "event create" ); ev.push_back( e ); }
	int64_t sent = 0;
	for( int k = 0; k < slices; ++k )
		{
		const int64_t f0 = frames_per_slice * k, f1 = std::min<int64_t>( F, f0 + frames_per_slice );
		// samples the frames below f1 read: up to hop * (f1 - 1) + W/2 (AudioPV.cpp:52)
		int64_t need = ( k == slices - 1 ) ? n : std::min<int64_t>( n, (int64_t) hop * ( f1 - 1 ) - W / 2 + W );
		if( need < sent ) need = sent;
		{ LaunchTimer lt( ctx, 9, ctx->h2d );
		  rc = copy_h2d_2d( ctx, d_audio + sent, sizeof( float ) * (size_t) n, h_audio + sent, sizeof( float ) * (size_t) n,
		                    sizeof( float ) * (size_t)( need - sent ), (size_t) C ); }
		if( rc ) return rc;
		sent = need;
		CK( cudaEventRecord( ev[k], ctx->h2d ), "event record" );
		CK( cudaStreamWaitEvent( ctx->compute, ev[k], 0 ), "stream wait" );
		if( f1 > f0 )
			{
			AnalysisCall a{ d_audio, n, 0, n, C, n, sr, W, hop, N, f0, f1, d_pv + 2 * f0 * B, F * (int64_t) B };
			rc = analysis_range( ctx, a );
			if( rc ) return rc;
			}
		if( cancelled( cancel ) ) return fail( ctx, FLAN_B200_CANCELLED, "cancelled" );
		}
	rc = side_release( ctx, ctx->h2d, d_audio );
	main_release( ctx, d_audio );
	main_release( ctx, d_pv );
	return rc;
	}

int flan_b200_convert_to_audio_d2h( flan_b200_ctx * ctx, const float * d_pv, int C, int64_t F, int B,
                                    float sr, float ar, int W, float * d_audio_out, float * h_audio_out,
                                    const volatile int * cancel, const volatile int ** nan_flag )
	{
	if( !ctx || !d_pv || !d_audio_out || !h_audio_out ) return FLAN_B200_INVALID;
	if( !( ar > 0.0f ) || !( sr > 0.0f ) ) return fail( ctx, FLAN_B200_INVALID, "rates must be positive" );
	const int hop = flan_b200_hop_from_rates( sr, ar );
	if( hop < 1 ) return fail( ctx, FLAN_B200_INVALID, "analysis_rate above sample_rate gives hop 0" );
	const int64_t out_n = F * hop;
	CallLock lock( ctx );
	if( find_block( ctx, d_pv ) && find_block( ctx, d_audio_out ) ) ctx->compute = ctx->s_syn;
	main_acquire( ctx, d_pv );
	main_acquire( ctx, d_audio_out );
	int rc = side_acquire( ctx, ctx->d2h, d_audio_out );       // an earlier download of this block, if any
	if( rc ) return rc;
	SynthCall s{ d_pv, F * B, C, 0, F, F, B, sr, ar, W };
	s.d_out = d_audio_out; s.out_stride = out_n; s.out_offset = 0; s.out_len = out_n; s.cancel = cancel;
	s.reuse_summary = take_promise( d_pv );
	const int slot = (int)( ctx->flag_next++ % flan_b200_ctx::FLAG_SLOTS );
	CK( cudaMemsetAsync( ctx->d_flags + slot, 0, sizeof( int ), ctx->compute ), "flag clear" );
	s.d_nan_flag = ctx->d_flags + slot;
	ctx->h_flags[slot] = 0;
	s.copy_bytes = sizeof( float ) * (size_t) C * out_n;
	std::vector<cudaEvent_t> & ev = ctx->slice_events;
	while( (int) ev.size() < 16 ) { cudaEvent_t e; CK( cudaEventCreateWithFlags( &e, cudaEventDisableTiming ), "event create" ); ev.push_back( e ); }
	int64_t got = 0;
	bool flag_sent = false;
	s.on_chunk = [&]( int k, int64_t done ) -> int
		{
		if( !flag_sent )
			{
			CK( cudaMemcpyAsync( ctx->h_flags + slot, ctx->d_flags + slot, sizeof( int ), cudaMemcpyDeviceToHost, ctx->compute ), "flag read" );
			flag_sent = true;
			}
		CK( cudaEventRecord( ev[k], ctx->compute ), "event record" );
		CK( cudaStreamWaitEvent( ctx->d2h, ev[k], 0 ), "copy stream wait" );
		if( done > got )
			{
			int rc2;
			{ LaunchTimer lt( ctx, 10, ctx->d2h );
			  rc2 = copy_d2h_2d( ctx, h_audio_out + got, sizeof( float ) * (size_t) out_n, d_audio_out + got, sizeof( float ) * (size_t) out_n,
			                     sizeof( float ) * (size_t)( done - got ), (size_t) C ); }
			if( rc2 ) return rc2;
			got = done;
			}
		return FLAN_B200_OK;
		};
	rc = synth_range( ctx, s );
	if( rc ) return rc;
	if( nan_flag ) *nan_flag = ctx->h_flags + slot;
	rc = side_release( ctx, ctx->d2h, d_audio_out );
	main_release( ctx, d_pv );
	main_release( ctx, d_audio_out );
	if( cancelled( cancel ) ) return fail( ctx, FLAN_B200_CANCELLED, "cancelled" );
	return rc;
	}

// The plain host-buffer forms: upload, transform, download, wait. Device blocks come from (and return to) the cache.
int flan_b200_convert_to_pv_host( flan_b200_ctx * ctx, const float * h_audio, int C, int64_t n,
                                  float sr, int W, int hop, int N, int mid_side,
                                  float * h_pv, const volatile int * cancel )
	{
	if( !ctx ) return FLAN_B200_INVALID;
	if( hop < 1 || C < 1 || n < 0 ) return fail( ctx, FLAN_B200_INVALID, "bad shape" );
	if( mid_side && C != 2 ) return fail( ctx, FLAN_B200_INVALID, "mid/side needs exactly two channels (AudioPV.cpp:82)" );
	const int64_t F = flan_b200_num_frames( n, hop );
	const int B = N / 2 + 1;
	const size_t audio_bytes = sizeof( float ) * (size_t) C * n;
	const size_t pv_bytes = sizeof( float ) * 2 * (size_t) C * F * B;
	float * d_audio = nullptr, * d_ms = nullptr, * d_pv = nullptr;
	int rc = flan_b200_malloc( ctx, audio_bytes, (void **) &d_audio );
	if( !rc && mid_side ) rc = flan_b200_malloc( ctx, audio_bytes, (void **) &d_ms );
	if( !rc ) rc = flan_b200_malloc( ctx, pv_bytes, (void **) &d_pv );
	if( !rc && !mid_side ) rc = flan_b200_convert_to_pv_h2d( ctx, h_audio, d_audio, C, n, sr, W, hop, N, d_pv, cancel );
	if( !rc && mid_side )
		{
		rc = flan_b200_upload( ctx, d_audio, h_audio, audio_bytes );
		if( !rc ) rc = flan_b200_mid_side( ctx, d_audio, d_ms, n );
		if( !rc ) rc = flan_b200_convert_to_pv( ctx, d_ms, C, n, sr, W, hop, N, d_pv, cancel );
		}
	if( !rc ) rc = flan_b200_download( ctx, h_pv, d_pv, pv_bytes );
	if( !rc ) rc = flan_b200_wait( ctx, d_pv );
	else flan_b200_synchronize( ctx );
	flan_b200_free( ctx, d_audio ); flan_b200_free( ctx, d_ms ); flan_b200_free( ctx, d_pv );
	return rc;
	}

int flan_b200_convert_to_audio_host( flan_b200_ctx * ctx, const float * h_pv, int C, int64_t F, int B,
                                     float sr, float ar, int W, int left_right,
                                     float * h_audio_out, const volatile int * cancel, int * nan_or_inf )
	{
	if( !ctx ) return FLAN_B200_INVALID;
	if( C < 1 || F < 0 || B < 2 || !( ar > 0.0f ) ) return fail( ctx, FLAN_B200_INVALID, "bad shape" );
	if( left_right && C != 2 ) return fail( ctx, FLAN_B200_INVALID, "left/right needs exactly two channels (AudioPV.cpp:143)" );
	const int hop = flan_b200_hop_from_rates( sr, ar );
	if( hop < 1 ) return fail( ctx, FLAN_B200_INVALID, "hop < 1" );
	const int64_t out_n = F * hop;
	const size_t pv_bytes = sizeof( float ) * 2 * (size_t) C * F * B;
	const size_t audio_bytes = sizeof( float ) * (size_t) C * out_n;
	float * d_pv = nullptr, * d_audio = nullptr, * d_lr = nullptr;
	const volatile int * flag = nullptr;
	int rc = flan_b200_malloc( ctx, pv_bytes, (void **) &d_pv );
	if( !rc ) rc = flan_b200_malloc( ctx, audio_bytes, (void **) &d_audio );
	if( !rc && left_right ) rc = flan_b200_malloc( ctx, audio_bytes, (void **) &d_lr );
	if( !rc ) rc = flan_b200_upload( ctx, d_pv, h_pv, pv_bytes );
	if( !rc && !left_right )
		{
		rc = flan_b200_convert_to_audio_d2h( ctx, d_pv, C, F, B, sr, ar, W, d_audio, h_audio_out, cancel, &flag );
		if( !rc ) rc = flan_b200_wait( ctx, d_audio );
		if( !rc && nan_or_inf ) *nan_or_inf = *flag;
		}
	if( !rc && left_right )
		{
		rc = flan_b200_convert_to_audio( ctx, d_pv, C, F, B, sr, ar, W, d_audio, cancel, nan_or_inf );
		if( !rc ) rc = flan_b200_mid_side( ctx, d_audio, d_lr, out_n );
		if( !rc ) rc = flan_b200_download( ctx, h_audio_out, d_lr, audio_bytes );
		if( !rc ) rc = flan_b200_wait( ctx, d_lr );
		}
	if( rc ) flan_b200_synchronize( ctx );
	flan_b200_free( ctx, d_pv ); flan_b200_free( ctx, d_audio ); flan_b200_free( ctx, d_lr );
	return rc;
	}

} // extern "C"
