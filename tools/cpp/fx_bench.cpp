// tools/cpp/fx_bench.cpp -- timing of the PV-domain methods with a Function written as a lambda and as an expression
// (flan/fx.h), for tools/fxbench.py. Each call is bracketed by a synchronise of the engine's device.
#include "flan/Audio/Audio.h"
#include "flan/PV/PV.h"
#include "flan/fx.h"
#include "flan_b200.h"

#include <chrono>
#include <memory>

using namespace flan;

namespace {

// op: 0 repitch, 1 stretch, 2 modify_frequency; cls: 0 constant, 1 time only, 2 frequency only, 3 both.
Function<TF, float> factor( int op, int cls, bool lambda )
	{
	using fx::t; using fx::f;
	if( cls == 0 ) return op == 2 ? 1000.0f : 1.25f;
	if( op < 2 )
		switch( cls )
			{
			case 1: if( lambda ) return []( TF x ) { return 1.0f + x.t / 3600.0f; }; return 1.0f + t / 3600.0f;
			case 2: if( lambda ) return []( TF x ) { return 1.0f + x.f / 96000.0f; }; return 1.0f + f / 96000.0f;
			default: if( lambda ) return []( TF x ) { return 1.0f + x.t / 7200.0f + x.f / 96000.0f; }; return 1.0f + t / 7200.0f + f / 96000.0f;
			}
	switch( cls )
		{
		case 1: if( lambda ) return []( TF x ) { return 1000.0f + x.t; }; return 1000.0f + t;
		case 2: if( lambda ) return []( TF x ) { return x.f * 0.8f + 30.0f; }; return f * 0.8f + 30.0f;
		default: if( lambda ) return []( TF x ) { return x.f * ( 1.0f + x.t / 3600.0f ); }; return f * ( 1.0f + t / 3600.0f );
		}
	}

std::unique_ptr<PV> g_pv;

}

extern "C" {

// Analyses one channel once and keeps its PV on the device for fx_bench_call. Returns frames or -1.
int fx_bench_setup( const float * audio, int n, float sr, int W, int hop, int N )
	{
	Audio a = Audio::create_from_buffer( std::vector<float>( audio, audio + size_t( n ) ), 1, sr );
	g_pv = std::make_unique<PV>( a.convert_to_PV( W, hop, N ) );
	if( g_pv->is_null() ) return -1;
	flan_b200_synchronize( b200::context() );
	return g_pv->get_num_frames();
	}

// Wall time of one call, synchronised before and after, in milliseconds; -1 on a null result.
double fx_bench_call( int op, int cls, int lambda )
	{
	const Function<TF, float> fn = factor( op, cls, lambda != 0 );
	flan_b200_synchronize( b200::context() );
	const auto t0 = std::chrono::steady_clock::now();
	PV out = op == 0 ? g_pv->repitch( fn ) : op == 1 ? g_pv->stretch( fn ) : g_pv->modify_frequency( fn );
	flan_b200_synchronize( b200::context() );
	const auto t1 = std::chrono::steady_clock::now();
	return out.is_null() ? -1.0 : std::chrono::duration<double, std::milli>( t1 - t0 ).count();
	}

void fx_bench_teardown( void ) { g_pv.reset(); }

}
