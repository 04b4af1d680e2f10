// flan_b200/csrc/pv_ctx.h -- the engine context behind the C ABI (include/flan_b200.h), shared by the pv_capi*.cu
// translation units. Host-side only: plan cache, device block cache with per-block ordering events, scratch workspace,
// copy streams with their pinned staging rings, the copy-thread pool, and the call lock.
//
// Concurrency contract (reference: Audio::convert_to_PV / PV::convert_to_audio are const and re-entrant, the only lock
// on the path is FFTW's planner mutex, FFTHelper.cpp:9,19): any entry point may be called from any host thread on the
// same context. A call holds `call_mutex` from its first to its last enqueue, so the multi-launch sequences that share
// the workspace never interleave; the error text is per calling thread.
#pragma once

#include "../../include/flan_b200.h"

#include "pv_launch.h"
#include "pv_modify.h"
#include "pv_io.h"
#include "pv_tables.h"
#include "pv_generic.h"

#include <cuda_runtime.h>

#include <condition_variable>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <optional>
#include <string>
#include <thread>
#include <tuple>
#include <vector>

namespace pvrt {

struct DevicePlan
	{
	pvk::HostTables host;
	float * win_analysis = nullptr;
	float * win_synthesis = nullptr;
	float * expected = nullptr;
	float2 * binc = nullptr;
	float2 * post_tw = nullptr;
	float2 * post_rot = nullptr;
	float4 * binc4 = nullptr;
	float2 * pass_tw = nullptr;
	float2 * pass_tw16 = nullptr;
	float2 * pass_tw_rev = nullptr;
	// dft sizes the templated kernels do not cover (pv_generic.cu): tables of the run-time-sized transform
	bool generic = false;
	pvk::GenericHost generic_host;
	pvk::GenericFft generic_fft{};
	float2 * g_tw = nullptr, * g_chirp = nullptr, * g_chirp_fft = nullptr;
	};

// One cudaMalloc'ed allocation handed out by flan_b200_malloc. Blocks are cached on free (never returned to the driver
// before flan_b200_destroy or an allocation failure), and carry the two events that order the context's stream against
// its copy streams: `main_event` follows the last use on the context's stream, `side_event` the last copy into or out of
// the block on a copy stream. Whoever touches the block next waits on exactly those, not on whole streams, so one
// caller's upload never queues behind another caller's kernels.
struct Block
	{
	void * ptr = nullptr;
	size_t bytes = 0;
	cudaEvent_t main_event = nullptr; bool main_pending = false; cudaStream_t main_stream = nullptr;
	cudaEvent_t side_event = nullptr; bool side_pending = false;
	};

// Fixed pool of host threads for staging copies between pageable memory and the pinned rings (a single thread moves
// ~14 GB/s, four ~48 GB/s on the GPU box's host: tools/micro/hostcopy.cu).
class CopyPool
	{
public:
	explicit CopyPool( int threads );
	~CopyPool();
	void copy( void * dst, const void * src, size_t bytes );       // returns when done
	int threads() const { return (int) workers_.size() + 1; }
private:
	struct Task { char * dst; const char * src; size_t bytes; };
	void run();
	std::vector<std::thread> workers_;
	std::mutex m_;
	std::condition_variable cv_, done_cv_;
	std::vector<Task> queue_;
	int outstanding_ = 0;
	bool stop_ = false;
	};

// Pinned staging ring of one copy direction: `depth` slices of `slice` bytes; slice i is free again once ev[i] has fired.
struct PinnedRing
	{
	char * base = nullptr;
	size_t slice = 0;
	int depth = 0;
	std::vector<cudaEvent_t> ev;
	std::vector<char> armed;
	int64_t next = 0;
	};

// The per-segment phase summaries at the head of the workspace (phase_layout) and the PV rows they describe. Three
// producers leave them for the next resynthesis of exactly those rows: the analysis kernel (flan_b200_hint_resynthesis),
// the bin-shared stretch gather (summary_window) and synth_range itself (flan_b200_phase_summary, then a _range call).
// One rule keeps the record true: get_workspace drops it on every call, so a consumer matches before it asks for the
// workspace (and forgets the match when get_workspace had to grow it: the old contents are gone), and a producer
// publishes after its launch. An entry point that writes PV rows without the workspace drops it.
struct PhaseSummaries
	{
	struct Key
		{
		const void * pv = nullptr; int64_t channel_stride = 0, frame_begin = 0, frame_end = 0;
		int C = 0, B = 0, W = 0, seg_len = 0;
		float sr = 0.0f, ar = 0.0f;             // compared bit for bit
		bool operator==( const Key & o ) const;
		};
	// what the producer left beside the summaries
	struct Source
		{
		bool needs_fix = false;     // entries marked by the analysis kernel (lowest bins, NaN / Inf): the next scan recomputes them
		bool nan_known = false;     // *nan_flag holds the NaN / Inf pre-scan result of these rows
		bool group_prefix = false;  // the scan scratch also holds the carry-free group prefixes of these summaries
		};
	int * nan_flag = nullptr;       // device int the producers raise for NaN / Inf in the rows they summarise
	int * sink = nullptr;           // device int for a pre-scan result nobody reads

	void publish( const Key & key, const Source & source );
	// What the producer of exactly these rows left, if the record holds them (and, with need_nan_flag, their NaN flag).
	std::optional<Source> match( const Key & key, bool need_nan_flag ) const;
	void drop();
	void drop_if_within( const Block & b );         // b is freed: summaries of rows inside it go
private:
	Key key_;
	Source source_;
	bool valid_ = false;
	};

} // namespace pvrt

struct flan_b200_ctx
	{
	int device = 0;
	int sms = 0;
	cudaStream_t stream = nullptr;          // the stream the device-pointer entry points enqueue on (flan_b200_set_stream)
	cudaStream_t compute = nullptr;         // the stream the call in progress enqueues its kernels on: `stream`, or one of:
	// The pipelined host-buffer forms run on streams of their own, analysis on s_ana and resynthesis on s_syn: a call whose
	// kernels wait for its upload must not hold up another caller's kernels queued behind it (head-of-line blocking on one
	// in-order stream cost a third of the end-to-end throughput with two callers). Blocks order the streams among
	// themselves (Block::main_event), the shared workspace through ws_event.
	cudaStream_t s_ana = nullptr, s_syn = nullptr;
	cudaStream_t h2d = nullptr, d2h = nullptr;   // copy streams of the host-buffer forms (non-blocking)
	// the first segment of a frame-range shard runs here, beside the rest of the shard on the calling stream (SynthCall::head_segments)
	cudaStream_t s_head = nullptr; cudaEvent_t head_fork = nullptr, head_join = nullptr;
	cudaEvent_t ws_event = nullptr; cudaStream_t ws_stream = nullptr; bool ws_recorded = false, ws_touched = false;
	int lock_depth = 0;
	std::recursive_mutex call_mutex;        // one call at a time enqueues on this context (see the header comment)
	std::map<std::tuple<int, int, int, uint32_t, uint32_t>, std::unique_ptr<pvrt::DevicePlan>> plans;
	void * workspace = nullptr;
	size_t workspace_bytes = 0;
	pvm::MapCheck * d_check = nullptr;      // time-map reduction of the PV-domain chain
	// NaN / Inf flags of the resynthesis pre-scan (AudioPV.cpp:88): a ring of slots, device side and pinned host side;
	// the two device ints after the ring are the summaries' flag and sink
	static constexpr int FLAG_SLOTS = 256;
	int * d_flags = nullptr;
	int * h_flags = nullptr;
	int64_t flag_next = 0;
	int64_t launches = 0;
	bool timing = false;
	pvrt::PhaseSummaries summaries;         // the phase summaries held in the workspace, and which rows they describe
	int max_seg_len = 0;                   // frames per CTA at most; 0 = by size (FLAN_B200_DEBUG builds: FLAN_B200_SEG_LEN)
#ifdef FLAN_B200_DEBUG
	// experiment knobs of development builds only (tools/experiments; pv_capi.cu: analysis_kernel / synthesis_kernel);
	// release builds carry the measured policy
	int tps_analysis = 0, pt_analysis = 0, one_buffer = -1, synth_variant = -1, tps_synthesis = 0, synth_one_buffer = -1;
#endif
	struct Timed { int kind; cudaEvent_t start, stop; };
	std::vector<Timed> timed;
	// device block cache
	std::map<uintptr_t, pvrt::Block> live;                  // by base address
	std::multimap<size_t, pvrt::Block> cached;              // free blocks by size
	size_t cached_bytes = 0;
	// host staging
	pvrt::PinnedRing ring_up, ring_down;
	std::unique_ptr<pvrt::CopyPool> copy_pool;
	std::vector<cudaEvent_t> slice_events;                  // per-slice events of the pipelined host forms (re-recorded call by call)
	};

namespace pvrt {

// ---- errors: per calling thread ------------------------------------------------------------------
std::string & thread_error();
int fail( flan_b200_ctx * ctx, int code, const std::string & msg );
int cuda_fail( flan_b200_ctx * ctx, cudaError_t e, const char * what );
#define CK( call, what ) do { cudaError_t e_ = ( call ); if( e_ != cudaSuccess ) return pvrt::cuda_fail( ctx, e_, what ); } while( 0 )

// Holds the context's call lock and makes its device current on the calling thread. The outermost lock of a call
// selects the stream its kernels go to (the context's stream; the pipelined host forms switch to s_ana / s_syn) and, on
// the way out, marks the point after the call's last use of the shared workspace.
struct CallLock
	{
	flan_b200_ctx * ctx;
	std::lock_guard<std::recursive_mutex> guard;
	explicit CallLock( flan_b200_ctx * c ) : ctx( c ), guard( c->call_mutex )
		{
		cudaSetDevice( ctx->device );
		if( ctx->lock_depth++ == 0 ) { ctx->compute = ctx->stream; ctx->ws_touched = false; }
		}
	~CallLock()
		{
		if( --ctx->lock_depth == 0 )
			{
			if( ctx->ws_touched ) { cudaEventRecord( ctx->ws_event, ctx->compute ); ctx->ws_stream = ctx->compute; ctx->ws_recorded = true; }
			ctx->compute = ctx->stream;
			}
		}
	CallLock( const CallLock & ) = delete;
	};

inline uint32_t fbits( float f ) { uint32_t u; std::memcpy( &u, &f, 4 ); return u; }
inline size_t align_up( size_t v, size_t a ) { return ( v + a - 1 ) / a * a; }
inline bool cancelled( const volatile int * cancel ) { return cancel && *cancel; }

int get_plan( flan_b200_ctx * ctx, int N, int W, int hop, float sr, float ar, DevicePlan ** out );
// The context's scratch area, at least `bytes` long. *kept (if given): the area was not reallocated, so what the last
// user left in it is still there.
int get_workspace( flan_b200_ctx * ctx, size_t bytes, void ** out, bool * kept = nullptr );
void free_plan( DevicePlan * p );

// Brackets one kernel launch with events when timing is on (bench.py's per-kernel roofline).
struct LaunchTimer
	{
	flan_b200_ctx * ctx; int kind; cudaStream_t stream; cudaEvent_t start = nullptr, stop = nullptr;
	LaunchTimer( flan_b200_ctx * c, int k, cudaStream_t on = nullptr );     // kinds >= 9: copies on a copy stream (not counted as launches)
	~LaunchTimer();
	};

// ---- block cache and cross-stream ordering ---------------------------------------------------------
Block * find_block( flan_b200_ctx * ctx, const void * p );             // block containing p, or null (foreign memory)
// The context's stream is about to read or write the block holding p: wait for copies in flight on it.
void main_acquire( flan_b200_ctx * ctx, const void * p );
// ... and has enqueued its last such access: remember the point for later copies.
void main_release( flan_b200_ctx * ctx, const void * p );
// A copy stream is about to touch the block holding p (foreign memory: orders against everything enqueued so far).
int side_acquire( flan_b200_ctx * ctx, cudaStream_t side, const void * p );
int side_release( flan_b200_ctx * ctx, cudaStream_t side, const void * p );

// RAII over one entry point: the context's stream waits for copies in flight on the blocks the call touches, and the
// point after its last enqueue is remembered on them.
struct BlockUse
	{
	flan_b200_ctx * ctx; const void * p[6]; int n = 0;
	BlockUse( flan_b200_ctx * c, std::initializer_list<const void *> ptrs ) : ctx( c )
		{
		for( const void * q : ptrs ) if( q && n < 6 && find_block( ctx, q ) ) { p[n++] = q; main_acquire( ctx, q ); }
		}
	~BlockUse() { for( int i = 0; i < n; ++i ) main_release( ctx, p[i] ); }
	BlockUse( const BlockUse & ) = delete;
	};

// ---- host staging ------------------------------------------------------------------------------------
bool host_is_pinned( const void * p );
int ensure_ring( flan_b200_ctx * ctx, PinnedRing & ring );
CopyPool & copy_pool( flan_b200_ctx * ctx );
// rows x width bytes between host (pitch h_pitch) and device (pitch d_pitch) on the given copy stream. Pinned host
// memory: one asynchronous 2-D copy. Pageable host memory: through the ring and the copy threads; an upload returns once
// the last slice is staged (still in flight), a download once the bytes are in h.
int copy_h2d_2d( flan_b200_ctx * ctx, void * d, size_t d_pitch, const void * h, size_t h_pitch, size_t width, size_t rows );
int copy_d2h_2d( flan_b200_ctx * ctx, void * h, size_t h_pitch, const void * d, size_t d_pitch, size_t width, size_t rows );

// ---- shared by the whole-signal, frame-range, pipelined and multi-device forms ---------------------------
struct SynthCall
	{
	const float * d_pv_rows; int64_t pv_channel_stride; int C;
	int64_t frame_begin, frame_end, frames_total; int B;
	float sr, ar; int W;
	const pvk::PhaseSeg * d_carry_in = nullptr; pvk::PhaseSeg * d_carry_out = nullptr;
	float * d_out = nullptr; int64_t out_stride = 0, out_offset = 0, out_len = 0;
	bool summary_only = false; bool reuse_summary = false;
	int seg_len = 0;                        // frames per CTA; 0: chosen from the local frame count
	const volatile int * cancel = nullptr;
	int * d_nan_flag = nullptr;             // device int the pre-scan raises; null: a scratch slot
	// pipelining: with on_chunk set the frames are launched in slices of whole waves of CTAs (at least 4 MiB of
	// copy_bytes each, 8 slices at most); after each slice on_chunk( k, sample_end ) is called with the absolute output
	// sample up to which the local span is final (every contribution enqueued)
	size_t copy_bytes = 0;
	std::function<int( int, int64_t )> on_chunk;
	// head_segments > 0 (multi-device forms): the first head_segments segments -- the frames whose windows reach into the
	// previous shard -- run as a launch of their own on the context's head stream, BESIDE the launch of all the other
	// segments (segments only meet in red.add's on pre-zeroed samples, so the two launches commute); head_event is
	// recorded on the head stream right after it, so the halo can travel while the interior computes. The calling
	// stream joins the head stream before synth_range returns.
	int head_segments = 0;
	cudaEvent_t head_event = nullptr;
	};
int synth_range( flan_b200_ctx * ctx, const SynthCall & s );
// Where synth_range keeps the phase scratch of a signal in the workspace: summaries [C][segs][B] at offset 0, then the
// accumulators entering each segment, then the scan's group states. A kernel that produces PV rows and leaves their
// summaries behind writes them there and publishes them (ctx->summaries).
struct PhaseLayout { int seg_len, segs, group_len, groups; size_t seg_bytes, acc_bytes, grp_bytes; size_t bytes() const { return seg_bytes + acc_bytes + grp_bytes; } };
PhaseLayout phase_layout( const flan_b200_ctx * ctx, int C, int64_t frames, int B, int W, int hop, int seg_len_given );
// Frames per segment of a resynthesis of `frames` frames with no length given: phase_layout's choice, and the length the
// multi-device forms cut a signal's shards at. Producer and consumer of summaries must agree on it, or the keys differ.
int resynthesis_seg_len( const flan_b200_ctx * ctx, int C, int64_t frames, int N, int W, int hop );
void promise_unchanged( const void * d_pv );
bool take_promise( const void * d_pv );
bool take_resynthesis_hint();
void set_resynthesis_hint();
// Slices of whole waves: CTAs per slice for `ctas` CTAs of a kernel with `wave` resident CTAs on the device.
int64_t ctas_per_slice( int64_t ctas, int64_t wave, size_t copy_bytes );

struct AnalysisCall
	{
	const float * d_audio_local; int64_t audio_stride, audio_offset, audio_len; int C; int64_t n_total;
	float sr; int W, hop, N;
	int64_t frame_begin, frame_end;
	float * d_pv_rows; int64_t pv_channel_stride;
	bool emit_summary = false;      // the rows will be resynthesised unchanged: also leave their phase summaries
	int emit_seg_len = 0;           // frame-range shards: the segment length of the WHOLE signal (0: this call is the whole signal)
	};
int analysis_range( flan_b200_ctx * ctx, const AnalysisCall & a );

// The time-map reduction of pvm::launch_map_check, read back (synchronises the calling stream): the output frame count
// of PV::modify_time (PVModify.cpp:312) and whether some column of the map descends.
int read_map_check( flan_b200_ctx * ctx, float sr, int hop, int64_t * out_frames, bool * descends );

} // namespace pvrt
