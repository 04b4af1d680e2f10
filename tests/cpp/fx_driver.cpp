// tests/cpp/fx_driver.cpp -- user code that passes expression Functions (flan/fx.h) to the PV-domain methods, next to
// the same calls with the lambda [&]( TF x ) { return e( x ); } of each expression. Exposed through extern "C" so that
// pytest can compare the two routes bit for bit, read the kernels each one reached and run them over several GPUs.
#include "flan/Audio/Audio.h"
#include "flan/PV/PV.h"
#include "flan/fx.h"

#include <cstring>

using namespace flan;

namespace {

Interpolator named( int id )
	{
	switch( id )
		{
		case 1: return Interpolator::midpoint();
		case 2: return Interpolator::nearest();
		case 3: return Interpolator::floor();
		case 4: return Interpolator::ceil();
		case 5: return Interpolator::smoothstep();
		case 6: return Interpolator::smootherstep();
		case 7: return Interpolator::sine();
		case 8: return Interpolator::sine2();
		case 9: return Interpolator::sqrt();
		default: return Interpolator::linear();
		}
	}

// op: 0 repitch, 1 stretch, 2 modify_time, 3 modify_frequency. cls: what the expression reads -- 0 neither, 1 t, 2 f,
// 3 both, 4 a curve of t (of f for modify_frequency). Exact ops only, and values that suit the op: factors for repitch /
// stretch, seconds for modify_time, Hz for modify_frequency. cls 1 and 2 of repitch / stretch are api_chain's kind 1.
fx::Expr expression( int op, int cls, int interp )
	{
	using fx::t; using fx::f;
	if( op <= 1 )
		switch( cls )
			{
			case 0: return fx::Expr( 1.25f ) + 0.25f;
			case 1: return 0.75f + 0.5f * t;
			case 2: return 1.0f + f / 24000.0f;
			case 3: return fx::max( 0.5f, 1.0f + f / 24000.0f - fx::floor( t * 4.0f ) / 8.0f + fx::where( t < 0.05f, 0.25f, 0.0f ) );
			default: return fx::curve( t, { { 0.0f, 1.0f }, { 0.05f, 1.5f }, { 0.1f, 0.8f }, { 0.2f, 1.2f } }, named( interp ) );
			}
	if( op == 2 )
		switch( cls )
			{
			case 0: return fx::Expr( 0.04f ) + 0.01f;
			case 1: return t * 1.25f + 0.01f;
			case 2: return 0.01f + f / 480000.0f;
			case 3: return t * ( 1.0f + f / 96000.0f );
			default: return fx::curve( t, { { 0.0f, 0.0f }, { 0.1f, 0.2f }, { 0.2f, 0.25f }, { 0.3f, 0.4f } }, named( interp ) );
			}
	switch( cls )
		{
		case 0: return fx::Expr( 1000.0f ) * 1.0f;
		case 1: return t * 1000.0f + 200.0f;
		case 2: return f * 0.8f + 30.0f;
		case 3: return f * ( 1.0f + t / 4.0f );
		default: return fx::curve( f, { { 0.0f, 0.0f }, { 4000.0f, 6000.0f }, { 24000.0f, 20000.0f } }, named( interp ) );
		}
	}

PV run( const PV & pv, int op, const Function<TF, float> & fn, int interp )
	{
	switch( op )
		{
		case 0: return pv.repitch( fn, named( interp ) );
		case 1: return pv.stretch( fn, named( interp ) );
		case 2: return pv.modify_time( fn, named( interp ) );
		default: return pv.modify_frequency( fn, named( interp ) );
		}
	}

int finish( const PV & out, float * pv_out, int * frames, float * audio_out )
	{
	if( out.is_null() ) return -1;
	*frames = out.get_num_frames();
	if( pv_out ) std::memcpy( pv_out, out.get_buffer().data(), sizeof( MF ) * out.get_buffer().size() );
	Audio a = out.convert_to_audio();
	if( a.is_null() ) return -1;
	if( audio_out ) std::memcpy( audio_out, a.get_buffer().data(), sizeof( float ) * a.get_buffer().size() );
	return a.get_num_frames();
	}

}

extern "C" {

// audio.convert_to_PV( W, hop, N ).<op>( expression or its lambda, interp ).convert_to_audio(). pv_out / audio_out may be
// null. *input_host_current: whether the input PV's host vector was made current by the call. Returns output samples per
// channel, or -1 on a null result.
int fx_chain( const float * audio, int C, int n, float sr, int W, int hop, int N, int op, int cls, int interp, int lambda,
              float * pv_out, int * frames, float * audio_out, int * input_host_current )
	{
	Audio a = Audio::create_from_buffer( std::vector<float>( audio, audio + size_t( C ) * n ), C, sr );
	PV pv = a.convert_to_PV( W, hop, N );
	if( pv.is_null() ) return -1;
	const fx::Expr e = expression( op, cls, interp );
	PV out = lambda ? run( pv, op, [&]( TF x ) { return e( x ); }, interp ) : run( pv, op, e, interp );
	*input_host_current = pv.storage().host_is_current() ? 1 : 0;
	return finish( out, pv_out, frames, audio_out );
	}

// The expression at one point, through Function<TF, float>::operator().
float fx_value( int op, int cls, int interp, float t, float f )
	{
	const Function<TF, float> fn( expression( op, cls, interp ) );
	return fn( TF{ t, f } );
	}

// Invalid expressions: a curve with a user-callable Interpolator, and one past the op limit. Returns 1 when both give a
// null PV from stretch and NaN from operator().
int fx_refusals( const float * audio, int n, float sr )
	{
	Audio a = Audio::create_from_buffer( std::vector<float>( audio, audio + size_t( n ) ), 1, sr );
	PV pv = a.convert_to_PV( 512, 128, 512 );
	if( pv.is_null() ) return -1;
	const fx::Expr user = fx::curve( fx::t, { { 0.0f, 1.0f }, { 1.0f, 2.0f } }, Interpolator( []( float x ) { return x * x; } ) );
	fx::Expr longer = fx::t;
	for( int i = 0; i < 40; ++i ) longer = longer + 1.0f;
	int ok = 1;
	for( const fx::Expr * e : { &user, const_cast<const fx::Expr *>( &longer ) } )
		ok &= !e->valid() && pv.stretch( *e ).is_null() && ( *e )( TF{ 0.0f, 0.0f } ) != ( *e )( TF{ 0.0f, 0.0f } );
	return ok;
	}

}
