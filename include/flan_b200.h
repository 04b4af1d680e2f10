/* include/flan_b200.h -- C ABI of the B200 phase-vocoder engine (libflan_b200.so).
 *
 * The reference (loganmcbroom/Flan) has no plugin or FFI seam for this path: the boundary is the C++
 * member call itself,
 *     PV    flan::Audio::convert_to_PV( Frame window, Frame hop, Frame dft, std::atomic<bool>& ) const
 *                                                   (src/flan/Audio/Audio.h:158-163, Conversions/AudioPV.cpp:12-78)
 *     Audio flan::PV::convert_to_audio( std::atomic<bool>& ) const
 *                                                   (src/flan/PV/PV.h:88-90,     Conversions/AudioPV.cpp:86-139)
 * plus the stereo wrappers convert_to_ms_PV / convert_to_lr_audio (AudioPV.cpp:80-84,141-145).
 * The entry points below are what a Flan build binds in place of the bodies of those four functions
 * (and of FFTHelper's FFTW plans, src/flan/FFTHelper.cpp:16-48); flan_b200/host/ holds the C++ side
 * (flan::Audio / flan::PV with the reference's signatures) and INTEGRATION.md the patch a maintainer
 * would apply. Plain pointers and sizes only; no C++ or torch types cross this line.
 *
 * Conventions
 *   - Layouts are the reference's: audio is planar float[C][n] (AudioBuffer.cpp:479-482); PV data is
 *     MF{float m; float f;} [C][F][B], B = dft/2+1 (PVBuffer.cpp:526-529). All offsets are 64-bit.
 *   - "d_" pointers are device memory on the context's GPU; "h_" pointers are host memory.
 *   - Device-pointer calls are asynchronous on the context's stream (flan_b200_set_stream) unless noted.
 *   - Every call returns FLAN_B200_OK or an error code; flan_b200_last_error() gives the text of the calling THREAD's
 *     last failure. The C++ layer maps any failure to the reference's "print and return a null object" (AudioPV.cpp:82,143).
 *   - Thread safety: like the reference's const conversions (re-entrant; FFTW's planner mutex, FFTHelper.cpp:9,19, is
 *     its only lock), every entry point may be called from any host thread on the same context. A call holds the
 *     context's call lock while it enqueues, so calls on one context are ordered, never interleaved; waiting
 *     (flan_b200_synchronize, flan_b200_wait) happens outside the lock.
 *   - There is no CPU fallback: without a CUDA device flan_b200_create() fails.
 *   - dft sizes: any size from 2 to 2^20 (FFTW plans any size, FFTHelper.cpp:16-26), window <= dft, hop >= 1. Powers of
 *     two from 256 to 8192 run the register-blocked kernels; every other size a run-time-sized transform (Stockham
 *     passes for powers of two, Bluestein otherwise) that is correct, not tuned. Sizes outside [2, 2^20] return
 *     FLAN_B200_UNSUPPORTED. For an odd dft size the bin frequencies and the inverse transform follow
 *     get_dft_size() = (num_bins - 1) * 2, as in the reference (PVBuffer.cpp:356-359).
 */
#ifndef FLAN_B200_H
#define FLAN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FLAN_B200_OK           0
#define FLAN_B200_INVALID      1   /* bad argument */
#define FLAN_B200_UNSUPPORTED  2   /* dft size outside the supported set */
#define FLAN_B200_CUDA         3   /* CUDA runtime error */
#define FLAN_B200_CANCELLED    4   /* cancel flag was raised (flan_CANCEL_POINT, defines.h:52-62) */
#define FLAN_B200_NOMEM        5

typedef struct flan_b200_ctx flan_b200_ctx;

/* Running-phase state of one (channel, bin) in split form: sum = q*P + r and its maximum prefix
 * (P = double(pi2)); see DESIGN.md "phase scan". Exchanged between frame-range shards. 32 bytes. */
typedef struct { double sum_q, sum_r, max_q, max_r; } flan_b200_phase_state;

/* ---- context ------------------------------------------------------------------------------- */
int  flan_b200_device_count( void );
int  flan_b200_create( int device, flan_b200_ctx ** out );
void flan_b200_destroy( flan_b200_ctx * ctx );
const char * flan_b200_last_error( const flan_b200_ctx * ctx );   /* ctx may be NULL: error of the last failed create */
int  flan_b200_set_stream( flan_b200_ctx * ctx, void * cuda_stream );   /* cudaStream_t; NULL = legacy default stream */
int  flan_b200_synchronize( flan_b200_ctx * ctx );                    /* the stream and both copy streams */
/* Waits until everything enqueued so far that touches the block holding d_ptr (kernels on the stream, copies on the copy
 * streams) has completed -- what a host accessor calls before it hands out the buffer's host copy. */
int  flan_b200_wait( flan_b200_ctx * ctx, const void * d_ptr );
/* The same for the copies only (uploads into / downloads out of the block): the host side of those copies is safe to
 * reuse afterwards; kernels that read or write the block may still be running. */
int  flan_b200_wait_copies( flan_b200_ctx * ctx, const void * d_ptr );
int  flan_b200_sm_count( const flan_b200_ctx * ctx );
/* Number of kernels this context has launched so far (bench.py reports it as gpu_launches). */
int64_t flan_b200_launch_count( const flan_b200_ctx * ctx );

/* Per-kernel device timing for bench.py's roofline line: when enabled, every kernel launch is bracketed by
 * CUDA events on the context's stream. flan_b200_kernel_time synchronises the stream, returns the summed
 * duration and launch count of one kernel kind since the last call for that kind, and resets it.
 * kinds: 0 analysis, 1 phase segment summary, 2 phase scan, 3 resynthesis, 4 mid/side + add + carry,
 * 5 repitch / modify_frequency, 6 stretch / modify_time, 7 table preparation and checks of the PV-domain chain, 8 file-format sample codecs. */
int flan_b200_set_timing( flan_b200_ctx * ctx, int enabled );
int flan_b200_kernel_time( flan_b200_ctx * ctx, int kind, double * total_ms, int64_t * launches );
/* Timeline of everything timed since timing was enabled: kind, start and stop in milliseconds relative to the first entry
 * (kinds as above, plus 9 = upload slice and 10 = download slice of the pipelined host-buffer forms). Synchronises the
 * device and consumes the entries; *count receives how many were written (at most capacity). */
int flan_b200_trace( flan_b200_ctx * ctx, int * kinds, double * start_ms, double * stop_ms, int capacity, int * count );

/* ---- device buffers (storage behind flan::AudioBuffer / flan::PVBuffer) ----------------------
 * Blocks are cached: flan_b200_free keeps the allocation for the next flan_b200_malloc of a similar size (no cudaMalloc /
 * cudaFree on the steady-state path); flan_b200_trim returns the cache to the driver. Each block remembers its last use
 * on the stream and on the copy streams, so copies and kernels on the same block are ordered against each other and
 * against nothing else. */
int flan_b200_malloc( flan_b200_ctx * ctx, size_t bytes, void ** d_out );
int flan_b200_free( flan_b200_ctx * ctx, void * d_ptr );
int flan_b200_trim( flan_b200_ctx * ctx );
/* Copies on the context's copy streams, ordered after / before the stream's work on the same block. Page-locked host
 * memory: asynchronous. Pageable host memory: staged through a pinned ring by a few copy threads -- an upload returns
 * once the last slice is staged, a download once the bytes have arrived. flan_b200_wait( d ) awaits either. */
int flan_b200_upload( flan_b200_ctx * ctx, void * d_dst, const void * h_src, size_t bytes );
int flan_b200_download( flan_b200_ctx * ctx, void * h_dst, const void * d_src, size_t bytes );
/* Page-lock a host range (a std::vector's storage) so that copies to and from it run asynchronously at PCIe speed.
 * Costs tens of milliseconds per 100 MB: worth it for buffers that are moved repeatedly. */
int flan_b200_host_register( flan_b200_ctx * ctx, void * h_ptr, size_t bytes );
int flan_b200_host_unregister( flan_b200_ctx * ctx, void * h_ptr );

/* ---- shapes (reference arithmetic) ---------------------------------------------------------- */
/* F = n / hop + 1 with an integer quotient (AudioPV.cpp:17). */
int64_t flan_b200_num_frames( int64_t n, int hop );
/* hop = int( sample_rate / analysis_rate ) (PVBuffer::get_hop_size, PVBuffer.cpp:381-384). */
int flan_b200_hop_from_rates( float sample_rate, float analysis_rate );
/* analysis_rate = float(sample_rate) / hop (AudioPV.cpp:25). */
float flan_b200_analysis_rate( float sample_rate, int hop );

/* ---- Audio::convert_to_PV (AudioPV.cpp:12-78) ----------------------------------------------- */
/* d_audio: float[C][n]; d_pv: MF[C][F][dft/2+1], F = flan_b200_num_frames(n, hop).
 * cancel (may be NULL) is the host-side flag of flan_CANCEL_ARG, polled between launches. */
int flan_b200_convert_to_pv( flan_b200_ctx * ctx, const float * d_audio, int channels, int64_t n,
                             float sample_rate, int window_size, int hop, int dft_size,
                             float * d_pv, const volatile int * cancel );

/* Frame-range shard of the same transform: produce frames [frame_begin, frame_end) of every channel.
 * d_audio_local holds, per channel (stride audio_stride elements), samples [audio_offset, audio_offset +
 * audio_len) of the signal and must cover [hop*(frame_begin-1) - window/2, hop*(frame_end-1) + window/2)
 * clipped to [0, n_total) -- i.e. a left halo of window/2 + hop and a right halo of window/2 samples.
 * d_pv_rows: row 0 of channel c is frame frame_begin; channels are pv_channel_stride MF elements apart. */
int flan_b200_convert_to_pv_range( flan_b200_ctx * ctx, const float * d_audio_local, int64_t audio_stride,
                                   int64_t audio_offset, int64_t audio_len, int channels, int64_t n_total,
                                   float sample_rate, int window_size, int hop, int dft_size,
                                   int64_t frame_begin, int64_t frame_end,
                                   float * d_pv_rows, int64_t pv_channel_stride );

/* ---- PV::convert_to_audio (AudioPV.cpp:86-139) ---------------------------------------------- */
/* d_pv: MF[C][F][B]; d_audio_out: float[C][F*hop], hop = flan_b200_hop_from_rates(sr, analysis_rate).
 * *nan_or_inf (may be NULL, host memory, written after an internal stream sync only if non-NULL)
 * reports the is_nan_or_inf() pre-scan of AudioPV.cpp:88; like the reference, conversion continues. */
int flan_b200_convert_to_audio( flan_b200_ctx * ctx, const float * d_pv, int channels, int64_t frames, int bins,
                                float sample_rate, float analysis_rate, int window_size,
                                float * d_audio_out, const volatile int * cancel, int * nan_or_inf );

/* Frame-range shard, step 1: phase state accumulated over the local frames [frame_begin, frame_end),
 * per (channel, bin): d_state_out[C][B]. Ranks all-gather these. */
int flan_b200_phase_summary( flan_b200_ctx * ctx, const float * d_pv_rows, int64_t pv_channel_stride,
                             int channels, int64_t frame_begin, int64_t frame_end, int bins,
                             float sample_rate, float analysis_rate, int window_size,
                             flan_b200_phase_state * d_state_out );
/* Step 2: state entering rank `rank` = combination of the gathered states of ranks 0..rank-1.
 * d_all: [ranks][C][B] in rank order; d_carry_out: [C][B]. */
int flan_b200_phase_carry( flan_b200_ctx * ctx, const flan_b200_phase_state * d_all, int rank,
                           int channels, int bins, flan_b200_phase_state * d_carry_out );
/* Step 3: resynthesise the local frames. d_out_local (ZEROED by this call) holds, per channel (stride
 * out_stride), samples [out_offset, out_offset + out_len) of the output; frames write the part of
 * [hop*frame_begin - window/2, hop*(frame_end-1) + window/2) that lies inside it and inside
 * [0, frames_total*hop). The first and last window-hop samples of that span are partial sums that the
 * caller adds to the neighbouring shard's (flan_b200_add). d_carry_in may be NULL (rank 0).
 * reuse_summary != 0 promises that the PV rows are unchanged since the flan_b200_phase_summary call that immediately
 * preceded on this context with the same rows / range / rates: its per-segment summaries (still in the context's
 * scratch) are reused instead of reading the PV data a second time. The promise is checked against the arguments. */
int flan_b200_convert_to_audio_range( flan_b200_ctx * ctx, const float * d_pv_rows, int64_t pv_channel_stride,
                                      int channels, int64_t frame_begin, int64_t frame_end, int64_t frames_total,
                                      int bins, float sample_rate, float analysis_rate, int window_size,
                                      const flan_b200_phase_state * d_carry_in, int reuse_summary,
                                      float * d_out_local, int64_t out_stride, int64_t out_offset, int64_t out_len );
/* The same with the frames whose windows reach into the previous shard launched first: head_event (a cudaEvent_t of the
 * caller, may be NULL) is recorded on the stream right after them, so that the window - hop partial sums at the head of
 * d_out_local can travel to the previous rank on another stream while the remaining frames compute. */
int flan_b200_convert_to_audio_range_head( flan_b200_ctx * ctx, const float * d_pv_rows, int64_t pv_channel_stride,
                                           int channels, int64_t frame_begin, int64_t frame_end, int64_t frames_total,
                                           int bins, float sample_rate, float analysis_rate, int window_size,
                                           const flan_b200_phase_state * d_carry_in, int reuse_summary,
                                           float * d_out_local, int64_t out_stride, int64_t out_offset, int64_t out_len,
                                           void * head_event );
/* ---- the two exchanges of sharded resynthesis between PROCESSES (one process per GPU, SURVEY 8e) ----------------------
 * Phase states and overlap-add halos travel as device-to-device copies over NVLink into mailboxes the peers opened through
 * CUDA IPC, ordered by sequence flags the receiving stream waits on (cuStreamWaitValue32): no kernel of the exchange
 * occupies an SM and nothing synchronises on the host. Every rank makes the same calls in the same order:
 *   create -> handle -> (all-gather the 64-byte handles by any means) -> connect, then per step
 *   state_slot -> flan_b200_phase_summary into it -> put_state -> get_states -> flan_b200_phase_carry -> release_states ->
 *   flan_b200_convert_to_audio_range_head -> put_halo (ranks > 0) -> add_halo (ranks < world - 1).
 * halo_samples: samples per channel of the largest halo (window - hop). Single-process callers use flan_b200_multi_*. */
#define FLAN_B200_IPC_HANDLE_BYTES 64
typedef struct flan_b200_exchange flan_b200_exchange;
int flan_b200_exchange_create( flan_b200_ctx * ctx, int rank, int world, int channels, int bins, int64_t halo_samples, flan_b200_exchange ** out );
void flan_b200_exchange_destroy( flan_b200_exchange * ex );
int flan_b200_exchange_handle( flan_b200_exchange * ex, void * handle64 );
int flan_b200_exchange_connect( flan_b200_exchange * ex, const void * handles /* world x 64 bytes, by rank */ );
/* where the next step's flan_b200_phase_summary should write this rank's state (pushed from there without a staging copy) */
int flan_b200_exchange_state_slot( flan_b200_exchange * ex, flan_b200_phase_state ** d_slot );
int flan_b200_exchange_put_state( flan_b200_exchange * ex, const flan_b200_phase_state * d_state );
int flan_b200_exchange_get_states( flan_b200_exchange * ex, const flan_b200_phase_state ** d_states /* [rank][channels][bins] */ );
int flan_b200_exchange_release_states( flan_b200_exchange * ex );
int flan_b200_exchange_put_halo( flan_b200_exchange * ex, const float * d_head, int64_t pitch, int channels, int64_t n, void * after_event );
int flan_b200_exchange_add_halo( flan_b200_exchange * ex, float * d_out, int64_t pitch, int channels, int64_t n );

/* d_out[i] += d_add[i], i < n (overlap-add halo received from a neighbour). */
int flan_b200_add( flan_b200_ctx * ctx, float * d_out, const float * d_add, int64_t n );

/* ---- Audio::convert_to_mid_side / convert_to_left_right (AudioConversions.cpp:32-56) --------- */
/* d_in, d_out: float[2][n]; the transform is its own inverse up to rounding. */
int flan_b200_mid_side( flan_b200_ctx * ctx, const float * d_in, float * d_out, int64_t n );

/* ---- PV-domain chain between analysis and resynthesis (BASELINE config 4) -------------------------------------
 * PV::repitch / PV::modify_frequency (src/flan/PV/PVModify.cpp:196-305, decl PV/PV.h:288-330) and PV::stretch /
 * PV::modify_time (PVModify.cpp:307-385, decl PV/PV.h:300-352) on device-resident PV data. Results are bit-identical
 * to the reference's float arithmetic for interpolators 0-6 and 9; 7 (sine) and 8 (sine2) evaluate cos / sin in
 * double and round, which differs from glibc's cosf in the last bit for a few inputs per thousand. Expression
 * Functions (flan_b200_fx_*, below) take the same approach for their transcendental ops, with the same caveat.
 *
 * The reference samples its Function<TF,float> argument over the frame x bin grid on the host (PV/PV.h:31-35);
 * here the sampled table arrives as a strided device view: element (frame, bin) = d_table[frame * frame_stride +
 * bin * bin_stride], strides (B,1) for a full float[F][B] table, (0,1) one row shared by every frame, (1,0) one
 * column shared by every bin, (0,0) a single value (what a constant Function samples to).
 * interp: 0 linear, 1 midpoint, 2 nearest, 3 floor, 4 ceil, 5 smoothstep, 6 smootherstep, 7 sine, 8 sine2, 9 sqrt
 * (the named constructors of Utility/Interpolator.cpp:15-101). d_pv_out must not alias d_pv. */

/* PV::repitch (PVModify.cpp:273-305): running sum of the factor along bins, bins -> Hz, lerp at every MF's own
 * frequency, then the scatter of modify_frequency_base. d_pv_out: MF[C][F][B]. */
int flan_b200_repitch( flan_b200_ctx * ctx, const float * d_pv, int channels, int64_t frames, int bins, float sample_rate,
                       const float * d_factor, int64_t factor_frame_stride, int factor_bin_stride,
                       int interp, float * d_pv_out );
/* modify_frequency_base (PVModify.cpp:196-257) behind PV::modify_frequency (:259-271): d_mod_hz is the mod function
 * sampled over the grid (Hz, strided view), d_in_mod float[C][F][B] the mod function evaluated by the caller at
 * (frame time, every MF's frequency) -- a user lambda of data on the host, PVModify.cpp:263-268. */
int flan_b200_modify_frequency( flan_b200_ctx * ctx, const float * d_pv, int channels, int64_t frames, int bins, float sample_rate,
                                const float * d_mod_hz, int64_t mod_frame_stride, int mod_bin_stride,
                                const float * d_in_mod, int interp, float * d_pv_out );
/* PV::stretch, first half (PVModify.cpp:373-382): running sum of the factor along frames, frames -> seconds.
 * d_map_out: dense float[F][B] when factor_bin_stride is 1, float[F] (a (1,0) view) when it is 0. */
int flan_b200_stretch_map( flan_b200_ctx * ctx, const float * d_factor, int64_t factor_frame_stride, int factor_bin_stride,
                           int64_t frames, int bins, float sample_rate, float analysis_rate, float * d_map_out );
/* Output frame count of modify_time_base for a time map in seconds: ceil( time_to_frame( maximum ) )
 * (PVModify.cpp:311-315). Synchronises the stream. A result <= 0 means an empty output. */
int flan_b200_modify_time_frames( flan_b200_ctx * ctx, const float * d_map, int64_t map_frame_stride, int map_bin_stride,
                                  int64_t frames, int bins, float sample_rate, float analysis_rate, int64_t * out_frames );
/* modify_time_base (PVModify.cpp:307-362) behind PV::modify_time (:364-369) and PV::stretch (:384).
 * d_pv_out: MF[C][out_frames][B], out_frames from flan_b200_modify_time_frames (checked). Synchronises once
 * internally: time maps that never descend run one thread per (channel, frame chunk, bin); others take the
 * reference's sequential walk per (channel, bin). */
int flan_b200_modify_time( flan_b200_ctx * ctx, const float * d_pv, int channels, int64_t frames, int bins,
                           float sample_rate, float analysis_rate,
                           const float * d_map, int64_t map_frame_stride, int map_bin_stride,
                           int interp, int64_t out_frames, float * d_pv_out, int summary_window );
/* summary_window > 0 (the PV's window size): when the time map is shared by all bins and never descends (PV::stretch with
 * a constant or time-only factor) the kernel walks its output frames in order and ALSO leaves behind the per-segment
 * phase summaries that flan_b200_convert_to_audio would otherwise compute with a second read of the rows. The context
 * holds the summaries of one set of rows at a time. They are dropped by the next call on this context that uses its
 * scratch space or writes PV rows, and by flan_b200_free of their buffer. A write by other means (a copy, a kernel of the
 * caller) is not seen. A caller that knows d_pv is unchanged since the call that produced it says so right before
 * resynthesis (same host thread): */
int flan_b200_promise_unchanged( flan_b200_ctx * ctx, const float * d_pv );
/* The producer can also be the analysis itself: after this hint (same host thread) the next flan_b200_convert_to_pv also
 * leaves the phase summaries of the rows it writes, for a caller that will resynthesise them as they are -- the round trip
 * of BASELINE configs 1-3. Full-window transforms of dft 2048 / 4096 / 8192 on long signals have that form (one
 * shared-memory word per bin: the increments of a bin lie within pi of its expected phase advance, and their differences
 * to it sum exactly in 32 bits); every other call ignores the hint. Costs ~10 % of the analysis kernel, saves the second
 * read of the rows (0.56 of 3.9 ms on cfg2). flan_b200_convert_to_pv_range consumes the hint too (a shard of a per-GPU
 * process: flan_b200_promise_unchanged before flan_b200_phase_summary then uses what it left). */
int flan_b200_hint_resynthesis( flan_b200_ctx * ctx );

/* ---- expression Functions: a Function<TF, float> as a program of t and f (flan/fx.h) ------------------------------
 * Postfix ops over a value stack, float constants and breakpoint curves. What a program depends on is known from its ops,
 * so it is sampled on the device into the compact view that dependence allows, and evaluated on the host by the same
 * source (flan_b200/csrc/pv_fx.cuh). Every node is one IEEE float32 operation with round to nearest, without contraction,
 * reassociation or folding, in the order of the ops. Operands: a binary op takes x (pushed first) and y (on top) and
 * pushes x op y; WHERE takes c, a, b and pushes c != 0 ? a : b; comparisons push 1.0f or 0.0f; MIN / MAX have fminf /
 * fmaxf semantics (a NaN operand yields the other one) with -0 < +0; ROUND is roundf (half away from zero). CURVE pops x
 * and pushes the envelope curve[index]: x <= x_0 gives y_0, x >= x_last gives y_last, NaN gives NaN, otherwise
 * y_i + interp( u ) * ( y_{i+1} - y_i ), u = ( x - x_i ) / ( x_{i+1} - x_i ), x_i <= x < x_{i+1}, interp one of the ids
 * 0-9 above. SIN, COS, EXP, LOG and POW compute ( float ) fn( ( double ) x ) on both sides; like interpolators 7 and 8
 * they are where host and device may differ: CUDA's and glibc's double results can round to different floats near a
 * tie. A NaN result is always the quiet NaN 0x7fc00000, on both sides (their hardware makes different NaN bits). Every
 * entry point validates the program (op codes, stack depth, a single result, curve indices, at least one
 * point per curve, finite and strictly ascending x, finite y, interpolator ids) and returns FLAN_B200_INVALID with a
 * message (flan_b200_fx_last_error) for a bad one. */
#define FLAN_B200_FX_MAX_OPS     64
#define FLAN_B200_FX_MAX_STACK   16
#define FLAN_B200_FX_MAX_CURVES  8
#define FLAN_B200_FX_MAX_POINTS  64
enum
	{
	FLAN_B200_FX_T, FLAN_B200_FX_F, FLAN_B200_FX_CONST,                                                     /* push */
	FLAN_B200_FX_ADD, FLAN_B200_FX_SUB, FLAN_B200_FX_MUL, FLAN_B200_FX_DIV, FLAN_B200_FX_MIN, FLAN_B200_FX_MAX,
	FLAN_B200_FX_LT, FLAN_B200_FX_LE, FLAN_B200_FX_GT, FLAN_B200_FX_GE, FLAN_B200_FX_EQ, FLAN_B200_FX_NE,
	FLAN_B200_FX_POW,                                                                                       /* x op y */
	FLAN_B200_FX_NEG, FLAN_B200_FX_ABS, FLAN_B200_FX_FLOOR, FLAN_B200_FX_CEIL, FLAN_B200_FX_ROUND, FLAN_B200_FX_SQRT,
	FLAN_B200_FX_SIN, FLAN_B200_FX_COS, FLAN_B200_FX_EXP, FLAN_B200_FX_LOG, FLAN_B200_FX_CURVE,              /* op x */
	FLAN_B200_FX_WHERE,                                                                                     /* c a b */
	FLAN_B200_FX_OP_COUNT
	};
typedef struct { int32_t code; int32_t index; float value; } flan_b200_fx_op;   /* value: CONST; index: CURVE */
typedef struct { int32_t points; int32_t interp; float x[FLAN_B200_FX_MAX_POINTS], y[FLAN_B200_FX_MAX_POINTS]; } flan_b200_fx_curve;
typedef struct flan_b200_fx_program
	{
	int32_t ops, curves;
	flan_b200_fx_op op[FLAN_B200_FX_MAX_OPS];
	flan_b200_fx_curve curve[FLAN_B200_FX_MAX_CURVES];
	} flan_b200_fx_program;
/* Validation and dependence: *uses_t / *uses_f (may be NULL) say whether the program reads t / f. */
int flan_b200_fx_check( const flan_b200_fx_program * prog, int * uses_t, int * uses_f );
/* Text of the calling thread's last failure of a flan_b200_fx_* call. */
const char * flan_b200_fx_last_error( void );
/* The host evaluation, the code the kernels run: *out = program( t, f ). */
int flan_b200_fx_eval( const flan_b200_fx_program * prog, float t, float f, float * out );
/* sample_function_over_domain (PV/PV.h:31-35) on the device: value( x, y ) = program( float( x ) * time_step,
 * float( y ) * bin_width ), with time_step = 1.0f / analysis_rate and bin_width = bin_to_frequency( 1 ), as PV::repitch
 * samples a lambda. Only what the program depends on is written: d_out receives frames * bins values (strides (bins, 1))
 * when it reads t and f, frames values (1, 0) for t alone, bins values (0, 1) for f alone, one value (0, 0) for neither:
 * the views of the PV-domain entry points above. flan_b200_fx_check tells the size in advance. Indices are 64-bit. */
int flan_b200_fx_sample( flan_b200_ctx * ctx, const flan_b200_fx_program * prog, int64_t frames, int bins,
                         float time_step, float bin_width, float * d_out, int64_t * frame_stride, int * bin_stride );
/* The program at every MF, as PV::modify_frequency evaluates its mod (PVModify.cpp:263-268): d_out[c][x][b] =
 * program( float( x ) / frame_rate, d_pv[c][x][b].f ) with frame_rate = float( sample_rate ) / float( hop )
 * (PVBuffer::frame_to_time). d_out: float[C][F][B], the d_in_mod of flan_b200_modify_frequency. */
int flan_b200_fx_at_pv( flan_b200_ctx * ctx, const flan_b200_fx_program * prog, const float * d_pv, int channels,
                        int64_t frames, int bins, float frame_rate, float * d_out );

/* ---- file formats either side of the path (SURVEY 8f-4) ---------------------------------------------------------
 * .flan RIFF-PV (PVBuffer::save / load, src/flan/PV/PVBuffer.cpp:99-140, 216-273; format described at
 * PV/PVBuffer.h:84-115): 24-bit signed samples, magnitude / dft size and frequency / sample rate, clamped to [-1,1],
 * times 2^23, truncated. Bit-identical to the reference's bytes. */
/* Sample codec on device buffers: count MF elements <-> 6 * count bytes (16-byte aligned). */
int flan_b200_flan_encode( flan_b200_ctx * ctx, const float * d_pv, int64_t count, float dft_size, float sample_rate, uint8_t * d_bytes );
int flan_b200_flan_decode( flan_b200_ctx * ctx, const uint8_t * d_bytes, int64_t count, float dft_size, float sample_rate, float * d_pv );
/* Whole files: header + samples streamed between the file and the device in chunks (synchronous). */
int flan_b200_save_flan( flan_b200_ctx * ctx, const char * path, const float * d_pv, int channels, int64_t frames, int bins,
                         float sample_rate, float analysis_rate, int window_size );
/* Header fields as PVBuffer::load reads them. *rate_field is the value load() stores as the analysis rate
 * (PVBuffer.cpp:245) -- which is the HOP that save() wrote there (:134): a reference quirk kept as is. */
int flan_b200_flan_info( flan_b200_ctx * ctx, const char * path, int * channels, int64_t * frames, int * bins,
                         float * sample_rate, float * rate_field, int * window_size );
int flan_b200_load_flan( flan_b200_ctx * ctx, const char * path, float * d_pv, int64_t capacity_mf );

/* WAV (RIFF, little-endian), as AudioBuffer::save / load handle it through libsndfile (src/flan/Audio/AudioBuffer.cpp:
 * 80-192; save defaults to PCM-24, :136). The sample types are libsndfile's for SF_FORMAT_WAV, and the codes below are
 * its sub-type values (SF_FORMAT_PCM_16 ...). libsndfile is external, not vendored, version unpinned: its default
 * conversions (normalisation on, clipping off) are restated. Write: clamp to [-1,1] (AudioBuffer.cpp:158-161; NaN passes
 * through), then
 *   PCM_U8  lrintf( x * 127 ) + 128        PCM_16  lrintf( x * 32767 )        PCM_24  lrintf( x * 8388607 )
 *   PCM_32  lrintf( x * 2^31 ), where +1.0 and NaN give 0x80000000 as on x86     FLOAT  the bits     DOUBLE  (double) x
 * (lrintf rounds half to even). Read: ( v - 128 ) / 128, v / 32768, v / 2^23, v / 2^31 (int -> float rounds to nearest
 * even), the bits, ( float ) d. The planar <-> interleaved reshuffle of AudioBuffer.cpp:122-125,152-155 is fused in.
 * Files read: format tag 1 (PCM, 1-4 byte containers), 3 (IEEE float, 32 or 64 bits) and WAVE_FORMAT_EXTENSIBLE with
 * the PCM or IEEE-float sub-format; the container width block_align / channels must be ceil( bits / 8 ) (20 valid bits in
 * 3 bytes read as PCM_24); anything else is FLAN_B200_UNSUPPORTED. Files written: PCM with the canonical 44-byte header,
 * FLOAT / DOUBLE with tag 3, an 18-byte fmt chunk and a fact chunk. Metadata strings are not carried, and a file over the
 * 4 GiB RIFF limit is refused before it is created. */
#define FLAN_B200_WAV_PCM_16  0x0002
#define FLAN_B200_WAV_PCM_24  0x0003
#define FLAN_B200_WAV_PCM_32  0x0004
#define FLAN_B200_WAV_PCM_U8  0x0005
#define FLAN_B200_WAV_FLOAT   0x0006
#define FLAN_B200_WAV_DOUBLE  0x0007
/* Sample codec on device buffers: planar float[channels][n] <-> interleaved frames, width( subtype ) * channels * n bytes
 * (16-byte aligned). */
int flan_b200_pcm_encode( flan_b200_ctx * ctx, const float * d_audio, int channels, int64_t n, int subtype, uint8_t * d_bytes );
int flan_b200_pcm_decode( flan_b200_ctx * ctx, const uint8_t * d_bytes, int channels, int64_t n, int subtype, float * d_audio );
/* The PCM_24 forms of the two above. */
int flan_b200_pcm24_encode( flan_b200_ctx * ctx, const float * d_audio, int channels, int64_t n, uint8_t * d_bytes );
int flan_b200_pcm24_decode( flan_b200_ctx * ctx, const uint8_t * d_bytes, int channels, int64_t n, float * d_audio );
/* Whole files: header + samples streamed between the file and the device in chunks (synchronous). save_wav writes
 * PCM_24, AudioBuffer::save's default. */
int flan_b200_save_wav_as( flan_b200_ctx * ctx, const char * path, const float * d_audio, int channels, int64_t n, float sample_rate,
                           int subtype );
int flan_b200_save_wav( flan_b200_ctx * ctx, const char * path, const float * d_audio, int channels, int64_t n, float sample_rate );
int flan_b200_wav_info( flan_b200_ctx * ctx, const char * path, int * channels, int64_t * n, float * sample_rate );
/* *subtype: the FLAN_B200_WAV_* code of the samples the file holds. */
int flan_b200_wav_format( flan_b200_ctx * ctx, const char * path, int * subtype );
int flan_b200_load_wav( flan_b200_ctx * ctx, const char * path, float * d_audio, int64_t capacity_samples );

/* ---- pipelined host-buffer forms: what flan::Audio::convert_to_PV / flan::PV::convert_to_audio call when the newest
 *      copy of the data is the object's host std::vector. --------------------------------------------------------
 * Analysis: h_audio (float[C][n]) is uploaded into d_audio (the object's device block) in a few slices on the copy
 * stream; the frames of each slice are transformed as soon as its samples have arrived. d_pv: MF[C][F][dft/2+1]. */
int flan_b200_convert_to_pv_h2d( flan_b200_ctx * ctx, const float * h_audio, float * d_audio, int channels, int64_t n,
                                 float sample_rate, int window_size, int hop, int dft_size,
                                 float * d_pv, const volatile int * cancel );
/* Resynthesis with the result prefetched to the host: the frames are transformed in a few slices, and the samples each
 * slice completes are copied into h_audio_out (float[C][F*hop]) on the download stream while the next slice computes.
 * Asynchronous when h_audio_out is page-locked; flan_b200_wait( ctx, d_audio_out ) awaits the download. *nan_flag (may
 * be NULL) receives a pointer to a pinned int that holds the is_nan_or_inf() result of AudioPV.cpp:88 once that wait
 * has returned (valid until 255 further calls). */
int flan_b200_convert_to_audio_d2h( flan_b200_ctx * ctx, const float * d_pv, int channels, int64_t frames, int bins,
                                    float sample_rate, float analysis_rate, int window_size,
                                    float * d_audio_out, float * h_audio_out,
                                    const volatile int * cancel, const volatile int ** nan_flag );

/* ---- plain host-buffer forms: upload, transform, download, wait (device blocks from the cache). ------------- */
int flan_b200_convert_to_pv_host( flan_b200_ctx * ctx, const float * h_audio, int channels, int64_t n,
                                  float sample_rate, int window_size, int hop, int dft_size, int mid_side,
                                  float * h_pv, const volatile int * cancel );
int flan_b200_convert_to_audio_host( flan_b200_ctx * ctx, const float * h_pv, int channels, int64_t frames, int bins,
                                     float sample_rate, float analysis_rate, int window_size, int left_right,
                                     float * h_audio_out, const volatile int * cancel, int * nan_or_inf );

/* ---- several GPUs of one box behind one handle (frame-range shards; SURVEY 8e) ------------------------------------
 * One process, one engine context per device. A signal is cut into contiguous frame ranges at multiples of the segment
 * length the uncut signal would use, so the result is the single-device result bit for bit. Analysis needs no exchange
 * (each shard is scattered with its halo of window/2 + hop samples on the left, window/2 on the right); resynthesis
 * moves the per-bin phase state (32 * channels * bins bytes per shard) and the window - hop overlap-add halo of every
 * shard boundary device to device (cudaMemcpyPeerAsync over NVLink), the halo behind the interior frames' compute.
 * Short signals use fewer shards than devices (a shard is at least one segment and 2 * ceil(window / hop) frames).
 * Between the two, repitch, and stretch / modify_time with a bin-shared map that never descends, keep the PV sharded
 * (flan_b200_multi_repitch / _stretch / _modify_time); other maps gather it onto device 0 and give a one-shard PV.
 * The structs are plain data owned by the caller; their device blocks come from the per-device contexts. */
#define FLAN_B200_MAX_DEVICES 16
typedef struct flan_b200_multi flan_b200_multi;
typedef struct
	{
	int channels; int64_t n;                      /* samples per channel of the whole signal */
	int shards;
	int64_t lo[FLAN_B200_MAX_DEVICES], hi[FLAN_B200_MAX_DEVICES];           /* shard i holds samples [lo, hi): float[channels][hi-lo] on device i */
	int64_t own_lo[FLAN_B200_MAX_DEVICES], own_hi[FLAN_B200_MAX_DEVICES];   /* of those, [own_lo, own_hi) are final (resynthesis output) */
	float * d[FLAN_B200_MAX_DEVICES];
	} flan_b200_sharded_audio;
typedef struct
	{
	int channels; int64_t frames; int bins;
	float sample_rate, analysis_rate; int window_size;
	int shards;
	int64_t frame_begin[FLAN_B200_MAX_DEVICES + 1];   /* shard i holds frames [frame_begin[i], frame_begin[i+1]): MF[channels][rows][bins] on device i */
	float * d[FLAN_B200_MAX_DEVICES];
	} flan_b200_sharded_pv;

/* devices == NULL: every visible device. A device may be listed more than once (tests on a single GPU). */
int  flan_b200_multi_create( const int * devices, int n_devices, flan_b200_multi ** out );
void flan_b200_multi_destroy( flan_b200_multi * m );
const char * flan_b200_multi_last_error( const flan_b200_multi * m );
int  flan_b200_multi_device_count( const flan_b200_multi * m );
flan_b200_ctx * flan_b200_multi_ctx( flan_b200_multi * m, int i );
int  flan_b200_multi_synchronize( flan_b200_multi * m );
/* Device timing across the handle (bench.py): begin synchronises and records a start event on every device's stream;
 * end records the stop events and returns the largest elapsed time of any device, in milliseconds. */
int  flan_b200_multi_time_begin( flan_b200_multi * m );
int  flan_b200_multi_time_end( flan_b200_multi * m, double * ms_max );
/* The frame ranges a signal of this shape is cut into: *shards and frame_begin[0 .. *shards]. */
int  flan_b200_multi_plan( const flan_b200_multi * m, int channels, int64_t n, int window_size, int hop, int dft_size,
                           int * shards, int64_t * frame_begin );
/* Host samples float[channels][n] -> every device's frame range with its halos (asynchronous for page-locked memory). */
int  flan_b200_multi_scatter_audio( flan_b200_multi * m, const float * h_audio, int channels, int64_t n,
                                    int window_size, int hop, int dft_size, flan_b200_sharded_audio * out );
/* Audio::convert_to_PV (AudioPV.cpp:12-78) over the shards. */
int  flan_b200_multi_convert_to_pv( flan_b200_multi * m, const flan_b200_sharded_audio * audio, float sample_rate,
                                    int window_size, int hop, int dft_size, flan_b200_sharded_pv * pv_out );
/* PV::convert_to_audio (AudioPV.cpp:86-139) over the shards, with the phase-state and halo exchange. */
int  flan_b200_multi_convert_to_audio( flan_b200_multi * m, const flan_b200_sharded_pv * pv, flan_b200_sharded_audio * audio_out );
/* flan_b200_hint_resynthesis and flan_b200_promise_unchanged for the sharded forms (same host thread): after the hint the
 * next flan_b200_multi_convert_to_pv also leaves every shard's phase summaries, in the segments of the whole signal; the
 * promise that pv is unchanged since then lets the next flan_b200_multi_convert_to_audio use them. */
int  flan_b200_multi_hint_resynthesis( flan_b200_multi * m );
int  flan_b200_multi_promise_unchanged( flan_b200_multi * m, const flan_b200_sharded_pv * pv );
/* Final samples of every shard -> host float[channels][n] (returns when the bytes have arrived). */
int  flan_b200_multi_gather_audio( flan_b200_multi * m, const flan_b200_sharded_audio * audio, float * h_audio );
/* PV rows of every shard -> host MF[channels][frames][bins] (h_pv, synchronous) and / or one device buffer of that layout
 * on device `to` of the handle (d_pv, asynchronous on that device's stream). Either pointer may be NULL. */
int  flan_b200_multi_gather_pv( flan_b200_multi * m, const flan_b200_sharded_pv * pv, float * h_pv, int to, float * d_pv );
/* The PV-domain chain over the shards (PV::repitch, PV::stretch, PV::modify_time): each reads pv, leaves it unchanged and
 * writes a new sharded PV into pv_out. Tables are HOST memory with the strides of the single-device forms: (bins,1),
 * (0,1), (1,0) or (0,0). Repitch: every device repitches its own rows with its rows of the table; pv_out has pv's frame
 * ranges. Stretch / modify_time with a map shared by all bins that never descends (a constant or time-only factor):
 * pv_out is cut like an analysed PV of its own frame count, each output shard is computed on its device from the input
 * rows it needs (read in place when the input shard on that device holds them, else peer-copied there), and leaves its
 * phase summaries, so that flan_b200_multi_promise_unchanged then lets flan_b200_multi_convert_to_audio skip the second
 * read of the rows. Any other map (per bin, or descending) gathers the PV onto device 0 and runs the single-device path
 * there: pv_out then has one shard. Either way the rows are the single-device result bit for bit. */
int  flan_b200_multi_repitch( flan_b200_multi * m, const flan_b200_sharded_pv * pv, const float * h_factor,
                              int64_t factor_frame_stride, int factor_bin_stride, int interp, flan_b200_sharded_pv * pv_out );
int  flan_b200_multi_stretch( flan_b200_multi * m, const flan_b200_sharded_pv * pv, const float * h_factor,
                              int64_t factor_frame_stride, int factor_bin_stride, int interp, flan_b200_sharded_pv * pv_out );
int  flan_b200_multi_modify_time( flan_b200_multi * m, const flan_b200_sharded_pv * pv, const float * h_map_seconds,
                                  int64_t map_frame_stride, int map_bin_stride, int interp, flan_b200_sharded_pv * pv_out );
int  flan_b200_multi_free_audio( flan_b200_multi * m, flan_b200_sharded_audio * audio );
int  flan_b200_multi_free_pv( flan_b200_multi * m, flan_b200_sharded_pv * pv );
/* What flan::Audio::convert_to_PV / flan::PV::convert_to_audio call for long signals when several GPUs are visible. */
int  flan_b200_multi_convert_to_pv_host( flan_b200_multi * m, const float * h_audio, int channels, int64_t n, float sample_rate,
                                         int window_size, int hop, int dft_size, flan_b200_sharded_pv * pv_out );
/* *nan_or_inf (may be NULL): the is_nan_or_inf() pre-scan of AudioPV.cpp:88 over all shards. */
int  flan_b200_multi_convert_to_audio_host( flan_b200_multi * m, const flan_b200_sharded_pv * pv, float * h_audio_out, int * nan_or_inf );

#ifdef __cplusplus
}
#endif
#endif
