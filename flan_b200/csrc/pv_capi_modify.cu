// flan_b200/csrc/pv_capi_modify.cu -- C ABI of the PV-domain chain between analysis and resynthesis (BASELINE config 4):
// PV::repitch / PV::modify_frequency / PV::stretch / PV::modify_time (reference PV/PVModify.cpp:196-385). Host-side
// orchestration only; the arithmetic is in pv_modify.cu.
#include "pv_ctx.h"

#include <cmath>

using namespace pvrt;

// ---- PV-domain chain (PV/PVModify.cpp:196-385) --------------------------------------------------

namespace {

int check_pv_shape( flan_b200_ctx * ctx, int C, int64_t F, int B, float sr, int interp )
	{
	if( C < 1 || F < 1 || B < 2 ) return fail( ctx, FLAN_B200_INVALID, "need channels >= 1, frames >= 1, bins >= 2" );
	if( !( sr > 0.0f ) ) return fail( ctx, FLAN_B200_INVALID, "sample_rate must be positive" );
	if( interp < 0 || interp > 9 ) return fail( ctx, FLAN_B200_INVALID, "interpolator id outside 0..9 (Utility/Interpolator.cpp)" );
	return FLAN_B200_OK;
	}

bool strides_ok( int64_t fs, int bs, int B ) { return ( bs == 0 || bs == 1 ) && ( fs == 0 || fs == ( bs ? B : 1 ) ); }

// mod_hz.frame_stride == 0 && bin_stride == 1 (one row of positions shared by all frames): plan + gather kernel, with
// the general row kernel as the device-side alternative when the plan kernel finds the positions non-monotone.
// plan_ws: 2 * B * 4 + 256 bytes of scratch for the plan, or null.
int repitch_common( flan_b200_ctx * ctx, const float * d_pv, int C, int64_t F, int B, float sr,
                    const pvm::Table & mod_hz, const float * d_in_mod, int interp, float * d_out, void * plan_ws )
	{
	pvm::RepitchArgs a{};
	a.pv = (const float2 *) d_pv; a.out = (float2 *) d_out;
	a.mod = mod_hz; a.in_mod = d_in_mod;
	a.F = F; a.B = B;
	a.bin_width = sr / float( ( B - 1 ) * 2 );                          // PVBuffer.cpp:438-441
	a.interp = interp;
	if( pvm::RepitchRow::bytes( B ) > 200 * 1024 ) return fail( ctx, FLAN_B200_UNSUPPORTED, "too many bins for one shared-memory row" );
	const int64_t rows = (int64_t) C * F;
	const int * skip_if = nullptr;
	if( plan_ws && mod_hz.frame_stride == 0 && mod_hz.bin_stride == 1 && pvm::repitch_shared_supported( B ) )
		{
		pvm::RepitchPlan plan{};
		plan.src = (int *) plan_ws; plan.mix = (float *)( plan.src + B ); plan.ok = (int *)( plan.mix + B );
		{ LaunchTimer lt( ctx, 7 ); CK( pvm::launch_repitch_plan( mod_hz.p, B, a.bin_width, interp, plan, ctx->compute ), "repitch plan launch" ); }
		{ LaunchTimer lt( ctx, 5 ); CK( pvm::launch_repitch_shared( a, plan, mod_hz.p, rows, ctx->sms, ctx->compute ), "repitch launch" ); }
		skip_if = plan.ok;
		}
	{ LaunchTimer lt( ctx, 5 ); CK( pvm::launch_repitch( a, rows, skip_if, ctx->compute ), "repitch launch" ); }
	return FLAN_B200_OK;
	}

size_t repitch_plan_bytes( int B ) { return align_up( sizeof( float ) * 2 * (size_t) B + sizeof( int ), 256 ); }

} // namespace

namespace pvrt {

// Reads the reduction back (synchronises the stream).
int read_map_check( flan_b200_ctx * ctx, float sr, int hop, int64_t * out_frames, bool * descends )
	{
	pvm::MapCheck h{};
	CK( cudaMemcpyAsync( &h, ctx->d_check, sizeof( h ), cudaMemcpyDeviceToHost, ctx->compute ), "map check read" );
	CK( cudaStreamSynchronize( ctx->compute ), "map check sync" );
	const float mx = pvm::key_float( h.max_key );
	const float last = std::ceil( mx * sr / float( hop ) );            // PVModify.cpp:312, PVBuffer.cpp:428-431
	*out_frames = (int64_t) pvm::to_int( last );                        // format.num_frames = last_output_frame (an int)
	*descends = h.descends != 0;
	return FLAN_B200_OK;
	}

} // namespace pvrt

extern "C" {

int flan_b200_repitch( flan_b200_ctx * ctx, const float * d_pv, int C, int64_t F, int B, float sr,
                       const float * d_factor, int64_t factor_frame_stride, int factor_bin_stride,
                       int interp, float * d_pv_out )
	{
	if( !ctx || !d_pv || !d_factor || !d_pv_out ) return FLAN_B200_INVALID;
	CallLock lock( ctx );
	BlockUse use( ctx, { d_pv, d_factor, d_pv_out } );
	int rc = check_pv_shape( ctx, C, F, B, sr, interp );
	if( rc ) return rc;
	if( !strides_ok( factor_frame_stride, factor_bin_stride, B ) )
		return fail( ctx, FLAN_B200_INVALID, "table strides must be (B,1), (0,1), (1,0) or (0,0)" );
	const int64_t rows = factor_frame_stride ? F : 1;
	void * ws = nullptr;
	const size_t hz_bytes = align_up( sizeof( float ) * (size_t) rows * B, 256 );
	rc = get_workspace( ctx, hz_bytes + repitch_plan_bytes( B ), &ws );
	if( rc ) return rc;
	const pvm::Table factor{ d_factor, factor_frame_stride, factor_bin_stride };
	{ LaunchTimer lt( ctx, 7 ); CK( pvm::launch_bin_prefix( factor, rows, B, sr, float( ( B - 1 ) * 2 ), (float *) ws, ctx->compute ), "repitch table launch" ); }
	const pvm::Table mod{ (const float *) ws, factor_frame_stride ? (int64_t) B : 0, 1 };
	return repitch_common( ctx, d_pv, C, F, B, sr, mod, nullptr, interp, d_pv_out, (char *) ws + hz_bytes );
	}

int flan_b200_modify_frequency( flan_b200_ctx * ctx, const float * d_pv, int C, int64_t F, int B, float sr,
                                const float * d_mod_hz, int64_t mod_frame_stride, int mod_bin_stride,
                                const float * d_in_mod, int interp, float * d_pv_out )
	{
	if( !ctx || !d_pv || !d_mod_hz || !d_in_mod || !d_pv_out ) return FLAN_B200_INVALID;
	CallLock lock( ctx );
	BlockUse use( ctx, { d_pv, d_mod_hz, d_in_mod, d_pv_out } );
	int rc = check_pv_shape( ctx, C, F, B, sr, interp );
	if( rc ) return rc;
	if( !strides_ok( mod_frame_stride, mod_bin_stride, B ) )
		return fail( ctx, FLAN_B200_INVALID, "table strides must be (B,1), (0,1), (1,0) or (0,0)" );
	const pvm::Table mod{ d_mod_hz, mod_frame_stride, mod_bin_stride };
	void * ws = nullptr;
	rc = get_workspace( ctx, repitch_plan_bytes( B ), &ws );
	if( rc ) return rc;
	return repitch_common( ctx, d_pv, C, F, B, sr, mod, d_in_mod, interp, d_pv_out, ws );
	}

int flan_b200_stretch_map( flan_b200_ctx * ctx, const float * d_factor, int64_t factor_frame_stride, int factor_bin_stride,
                           int64_t F, int B, float sr, float ar, float * d_map_out )
	{
	if( !ctx || !d_factor || !d_map_out ) return FLAN_B200_INVALID;
	CallLock lock( ctx );
	BlockUse use( ctx, { d_factor, d_map_out } );
	if( F < 1 || B < 2 || !( sr > 0.0f ) || !( ar > 0.0f ) ) return fail( ctx, FLAN_B200_INVALID, "bad shape or rates" );
	if( !strides_ok( factor_frame_stride, factor_bin_stride, B ) )
		return fail( ctx, FLAN_B200_INVALID, "table strides must be (B,1), (0,1), (1,0) or (0,0)" );
	const int hop = flan_b200_hop_from_rates( sr, ar );
	if( hop < 1 ) return fail( ctx, FLAN_B200_INVALID, "hop < 1" );
	const int cols = factor_bin_stride ? B : 1;
	const pvm::Table factor{ d_factor, factor_frame_stride, factor_bin_stride };
	void * ws = nullptr;
	const bool constant = factor_frame_stride == 0 && factor_bin_stride == 0;
	int rc = get_workspace( ctx, constant ? pvm::constant_prefix_scratch_bytes() : sizeof( float ) * (size_t) F * cols, &ws );
	if( rc ) return rc;
	LaunchTimer lt( ctx, 7 );
	if( constant )      // closed form per binade instead of F dependent additions
		CK( pvm::launch_constant_prefix( d_factor, F, sr / float( hop ), ws, d_map_out, ctx->sms, ctx->compute ), "stretch map launch" );
	else
		CK( pvm::launch_frame_prefix( factor, F, cols, sr / float( hop ), (float *) ws, d_map_out, ctx->sms, ctx->compute ), "stretch map launch" );
	ctx->launches += 1;
	return FLAN_B200_OK;
	}

int flan_b200_modify_time_frames( flan_b200_ctx * ctx, const float * d_map, int64_t map_frame_stride, int map_bin_stride,
                                  int64_t F, int B, float sr, float ar, int64_t * out_frames )
	{
	if( !ctx || !d_map || !out_frames ) return FLAN_B200_INVALID;
	CallLock lock( ctx );
	BlockUse use( ctx, { d_map } );
	if( F < 1 || B < 2 || !( sr > 0.0f ) || !( ar > 0.0f ) ) return fail( ctx, FLAN_B200_INVALID, "bad shape or rates" );
	if( !strides_ok( map_frame_stride, map_bin_stride, B ) )
		return fail( ctx, FLAN_B200_INVALID, "table strides must be (B,1), (0,1), (1,0) or (0,0)" );
	const int hop = flan_b200_hop_from_rates( sr, ar );
	if( hop < 1 ) return fail( ctx, FLAN_B200_INVALID, "hop < 1" );
	const pvm::Table mod{ d_map, map_frame_stride, map_bin_stride };
	{ LaunchTimer lt( ctx, 7 ); CK( pvm::launch_map_check( mod, map_frame_stride ? F : 1, map_bin_stride ? B : 1, ctx->d_check, ctx->sms, ctx->compute ), "map check launch" ); }
	bool descends = false;
	return read_map_check( ctx, sr, hop, out_frames, &descends );
	}

int flan_b200_modify_time( flan_b200_ctx * ctx, const float * d_pv, int C, int64_t F, int B, float sr, float ar,
                           const float * d_map, int64_t map_frame_stride, int map_bin_stride,
                           int interp, int64_t out_frames, float * d_pv_out, int summary_window )
	{
	if( !ctx || !d_pv || !d_map ) return FLAN_B200_INVALID;
	CallLock lock( ctx );
	BlockUse use( ctx, { d_pv, d_map, d_pv_out } );
	int rc = check_pv_shape( ctx, C, F, B, sr, interp );
	if( rc ) return rc;
	if( !( ar > 0.0f ) ) return fail( ctx, FLAN_B200_INVALID, "analysis_rate must be positive" );
	if( !strides_ok( map_frame_stride, map_bin_stride, B ) )
		return fail( ctx, FLAN_B200_INVALID, "table strides must be (B,1), (0,1), (1,0) or (0,0)" );
	const int hop = flan_b200_hop_from_rates( sr, ar );
	if( hop < 1 ) return fail( ctx, FLAN_B200_INVALID, "hop < 1" );
	const pvm::Table mod{ d_map, map_frame_stride, map_bin_stride };
	// The frame count and the choice between the parallel and the sequential walk both come from the map itself.
	{ LaunchTimer lt( ctx, 7 ); CK( pvm::launch_map_check( mod, map_frame_stride ? F : 1, map_bin_stride ? B : 1, ctx->d_check, ctx->sms, ctx->compute ), "map check launch" ); }
	int64_t frames = 0; bool descends = false;
	rc = read_map_check( ctx, sr, hop, &frames, &descends );
	if( rc ) return rc;
	if( frames != out_frames )
		return fail( ctx, FLAN_B200_INVALID, "out_frames does not match the map: expected " + std::to_string( frames ) );
	if( out_frames <= 0 ) return FLAN_B200_OK;
	if( !d_pv_out ) return FLAN_B200_INVALID;

	pvm::StretchArgs a{};
	a.pv = (const float2 *) d_pv; a.out = (float2 *) d_pv_out; a.mod = mod;
	a.F = F; a.out_frames = out_frames; a.B = B;
	a.sample_rate = sr; a.hop = float( hop ); a.interp = interp;
	a.pv_channel_stride = F * B; a.out_channel_stride = out_frames * B;
	a.chunk = 32;
	a.chunks = ( F - 1 + a.chunk - 1 ) / a.chunk;
	if( a.chunks < 1 ) a.chunks = 1;
	if( !descends && map_bin_stride == 0 && F < 0x7fffffff && out_frames < 0x7fffffff )
		{
		// one geometry for every bin: plan it once, then only the per-bin arithmetic remains -- as a gather by segments of
		// output frames, in the order resynthesis accumulates phase, so that with summary_window > 0 the kernel also leaves
		// the phase summaries of its output where flan_b200_convert_to_audio looks for them (flan_b200_promise_unchanged)
		const int W = summary_window > 0 ? summary_window : ( B - 1 ) * 2;
		const PhaseLayout lay = phase_layout( ctx, C, out_frames, B, W, hop, 0 );
		DevicePlan * dp = nullptr;
		if( summary_window > 0 ) { rc = get_plan( ctx, ( B - 1 ) * 2, W, hop, sr, ar, &dp ); if( rc ) return rc; }
		void * ws = nullptr;
		const size_t xpos_bytes = align_up( sizeof( int ) * (size_t) F, 256 ), mix_bytes = align_up( sizeof( float ) * (size_t) out_frames, 256 );
		const size_t phase_bytes = summary_window > 0 ? lay.bytes() : 0;
		rc = get_workspace( ctx, phase_bytes + xpos_bytes + mix_bytes + sizeof( int ) * (size_t) out_frames, &ws );
		if( rc ) return rc;
		char * base = (char *) ws + phase_bytes;
		pvm::StretchPlan plan{ (int *) base, (float *)( base + xpos_bytes ), (int *)( base + xpos_bytes + mix_bytes ) };
		pvm::StretchSummary summ{};
		summ.seg_len = lay.seg_len; summ.segs_per_channel = lay.segs;
		if( summary_window > 0 )
			{
			summ.seg_out = (pvk::PhaseSeg *) ws;
			summ.nan_flag = ctx->summaries.nan_flag;
			summ.k = dp->host.k; summ.P = dp->host.P; summ.rcpP = dp->host.rcpP;
			CK( cudaMemsetAsync( summ.nan_flag, 0, sizeof( int ), ctx->compute ), "flag clear" );
			}
		{ LaunchTimer lt( ctx, 6 ); CK( pvm::launch_stretch_planned( a, plan, summ, C, ctx->compute ), "stretch launch" ); ctx->launches++; }
		if( summary_window > 0 )
			ctx->summaries.publish( { d_pv_out, out_frames * B, 0, out_frames, C, B, W, lay.seg_len, sr, ar }, { /* needs_fix */ false, /* nan_known */ true } );
		}
	else
		{
		ctx->summaries.drop();          // these walks write the rows without the workspace: no summaries describe them
		if( !descends )
			{ LaunchTimer lt( ctx, 6 ); CK( pvm::launch_stretch_parallel( a, C, ctx->compute ), "stretch launch" ); }
		else
			{
			CK( cudaMemsetAsync( d_pv_out, 0, sizeof( float2 ) * (size_t) C * out_frames * B, ctx->compute ), "output clear" );   // PVModify.cpp:317-318
			LaunchTimer lt( ctx, 6 ); CK( pvm::launch_stretch_sequential( a, C, ctx->compute ), "stretch launch" );
			}
		}
	return FLAN_B200_OK;
	}

} // extern "C"
