// flan_b200/csrc/pv_capi_fx.cu -- C ABI of the expression Functions (include/flan_b200.h, flan_b200_fx_*): validation,
// the host evaluation (pv_fx.cuh's fx_eval, compiled here for the host without contraction) and the two device launches.
#include "pv_ctx.h"
#include "pv_fx.h"

#include <cmath>

using namespace pvrt;

namespace {

int fx_fail( const std::string & msg ) { thread_error() = msg; return FLAN_B200_INVALID; }

// Everything fx_eval relies on: known op codes, a stack that never underflows or exceeds its depth and ends with one
// value, curve indices in range, curves with 1 to FLAN_B200_FX_MAX_POINTS finite points in strictly ascending x, named
// interpolators.
int validate( const flan_b200_fx_program * p, int * uses_t, int * uses_f )
	{
	if( !p ) return fx_fail( "null program" );
	if( p->ops < 1 || p->ops > FLAN_B200_FX_MAX_OPS ) return fx_fail( "program needs 1 to " + std::to_string( FLAN_B200_FX_MAX_OPS ) + " ops" );
	if( p->curves < 0 || p->curves > FLAN_B200_FX_MAX_CURVES ) return fx_fail( "program has 0 to " + std::to_string( FLAN_B200_FX_MAX_CURVES ) + " curves" );
	for( int c = 0; c < p->curves; ++c )
		{
		const flan_b200_fx_curve & k = p->curve[c];
		const std::string at = "curve " + std::to_string( c ) + ": ";
		if( k.points < 1 || k.points > FLAN_B200_FX_MAX_POINTS ) return fx_fail( at + "needs 1 to " + std::to_string( FLAN_B200_FX_MAX_POINTS ) + " points" );
		if( k.interp < 0 || k.interp > 9 ) return fx_fail( at + "interpolator id outside 0..9 (only the named Interpolators)" );
		for( int i = 0; i < k.points; ++i )
			{
			if( !std::isfinite( k.x[i] ) || !std::isfinite( k.y[i] ) ) return fx_fail( at + "point " + std::to_string( i ) + " is not finite" );
			if( i > 0 && !( k.x[i - 1] < k.x[i] ) ) return fx_fail( at + "x must ascend strictly (point " + std::to_string( i ) + ")" );
			}
		}
	bool t = false, f = false;
	int depth = 0;
	for( int i = 0; i < p->ops; ++i )
		{
		const flan_b200_fx_op & o = p->op[i];
		const std::string at = "op " + std::to_string( i ) + ": ";
		int pops, pushes = 1;
		if( o.code < 0 || o.code >= FLAN_B200_FX_OP_COUNT ) return fx_fail( at + "unknown op code " + std::to_string( o.code ) );
		if( o.code <= FLAN_B200_FX_CONST ) pops = 0;
		else if( o.code <= FLAN_B200_FX_POW ) pops = 2;
		else if( o.code <= FLAN_B200_FX_CURVE ) pops = 1;
		else pops = 3;
		if( depth < pops ) return fx_fail( at + "stack underflow" );
		depth += pushes - pops;
		if( depth > FLAN_B200_FX_MAX_STACK ) return fx_fail( at + "stack deeper than " + std::to_string( FLAN_B200_FX_MAX_STACK ) );
		if( o.code == FLAN_B200_FX_CURVE && ( o.index < 0 || o.index >= p->curves ) ) return fx_fail( at + "curve index out of range" );
		t |= o.code == FLAN_B200_FX_T;
		f |= o.code == FLAN_B200_FX_F;
		}
	if( depth != 1 ) return fx_fail( "program leaves " + std::to_string( depth ) + " values, not one" );
	if( uses_t ) *uses_t = t;
	if( uses_f ) *uses_f = f;
	return FLAN_B200_OK;
	}

} // namespace

extern "C" {

int flan_b200_fx_check( const flan_b200_fx_program * prog, int * uses_t, int * uses_f ) { return validate( prog, uses_t, uses_f ); }

const char * flan_b200_fx_last_error( void ) { return thread_error().c_str(); }

int flan_b200_fx_eval( const flan_b200_fx_program * prog, float t, float f, float * out )
	{
	if( !out ) return fx_fail( "null output" );
	const int rc = validate( prog, nullptr, nullptr );
	if( rc ) return rc;
	*out = pvfx::fx_eval( *prog, t, f );
	return FLAN_B200_OK;
	}

int flan_b200_fx_sample( flan_b200_ctx * ctx, const flan_b200_fx_program * prog, int64_t F, int B,
                         float time_step, float bin_width, float * d_out, int64_t * frame_stride, int * bin_stride )
	{
	if( !ctx || !d_out || !frame_stride || !bin_stride ) return FLAN_B200_INVALID;
	int ut = 0, uf = 0;
	int rc = validate( prog, &ut, &uf );
	if( rc ) return rc;
	if( F < 1 || B < 1 ) return fail( ctx, FLAN_B200_INVALID, "need frames >= 1, bins >= 1" );
	CallLock lock( ctx );
	BlockUse use( ctx, { d_out } );
	const int64_t total = ( ut ? F : 1 ) * ( uf ? B : 1 );
	*frame_stride = ut ? ( uf ? B : 1 ) : 0;
	*bin_stride = uf ? 1 : 0;
	{ LaunchTimer lt( ctx, 7 ); CK( pvfx::launch_fx_sample( *prog, total, B, ut, uf, time_step, bin_width, d_out, ctx->sms, ctx->compute ), "fx sample launch" ); }
	return FLAN_B200_OK;
	}

int flan_b200_fx_at_pv( flan_b200_ctx * ctx, const flan_b200_fx_program * prog, const float * d_pv, int C,
                        int64_t F, int B, float frame_rate, float * d_out )
	{
	if( !ctx || !d_pv || !d_out ) return FLAN_B200_INVALID;
	int rc = validate( prog, nullptr, nullptr );
	if( rc ) return rc;
	if( C < 1 || F < 1 || B < 1 ) return fail( ctx, FLAN_B200_INVALID, "need channels >= 1, frames >= 1, bins >= 1" );
	CallLock lock( ctx );
	BlockUse use( ctx, { d_pv, d_out } );
	{ LaunchTimer lt( ctx, 7 ); CK( pvfx::launch_fx_at_pv( *prog, d_pv, (int64_t) C * F * B, F, B, frame_rate, d_out, ctx->sms, ctx->compute ), "fx at-PV launch" ); }
	return FLAN_B200_OK;
	}

} // extern "C"
