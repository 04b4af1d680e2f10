// PV-domain methods of the B200 build: PV::repitch, PV::stretch, PV::modify_time, PV::modify_frequency with the
// reference's signatures (src/flan/PV/PV.h:276-310, bodies PV/PVModify.cpp:196-385). The host does what only the host
// can do -- call the user's Function over the frame x bin grid (PV.h:31-35, Function.h:155-171) -- and the C ABI of
// libflan_b200.so (include/flan_b200.h) does the arithmetic on the device-resident PV data. An expression Function
// (flan/fx.h) is sampled on the device instead, into the compact table its dependence allows.
#include "flan/PV/PV.h"

#include <algorithm>
#include <iostream>
#include <optional>
#include <thread>
#include <vector>

#include "flan_b200.h"

namespace flan {

// ---- Interpolator: the named constructors of Utility/Interpolator.cpp:15-101 -----------------------------------
namespace { const float interp_pi = std::acos( -1.0f ); const float interp_sqrt2 = std::sqrt( 2.0f ); }

Interpolator Interpolator::linear()       { return Interpolator( Function<float, float>( []( float x ) { return x; } ), 0 ); }
Interpolator Interpolator::midpoint()     { return Interpolator( Function<float, float>( []( float ) { return 0.5f; } ), 1 ); }
Interpolator Interpolator::nearest()      { return Interpolator( Function<float, float>( []( float x ) { return std::round( x ); } ), 2 ); }
Interpolator Interpolator::floor()        { return Interpolator( Function<float, float>( []( float ) { return 0.0f; } ), 3 ); }
Interpolator Interpolator::ceil()         { return Interpolator( Function<float, float>( []( float ) { return 1.0f; } ), 4 ); }
Interpolator Interpolator::smoothstep()   { return Interpolator( Function<float, float>( []( float x ) { return x * x * ( 3.0f - 2.0f * x ); } ), 5 ); }
Interpolator Interpolator::smootherstep() { return Interpolator( Function<float, float>( []( float x ) { return x * x * x * ( x * ( x * 6.0f - 15.0f ) + 10.0f ); } ), 6 ); }
Interpolator Interpolator::sine()         { return Interpolator( Function<float, float>( []( float x ) { return ( 1.0f - std::cos( interp_pi * x ) ) / 2.0f; } ), 7 ); }
Interpolator Interpolator::sine2()        { return Interpolator( Function<float, float>( []( float x ) { return float( interp_sqrt2 * sin( interp_pi / 4.0f * x ) ); } ), 8 ); }
Interpolator Interpolator::sqrt()         { return Interpolator( Function<float, float>( []( float x ) { return std::sqrt( x ); } ), 9 ); }

namespace {

// A Function<TF, float> sampled over the PV's grid, on the device: the strided view include/flan_b200.h describes.
struct DeviceTable
	{
	b200::Mirror<float> data;
	const float * d = nullptr;
	int64_t frame_stride = 0;
	int bin_stride = 0;
	};

template<class Body> void for_rows( ExecutionPolicy policy, Frame rows, Body body )
	{
	unsigned workers = 1;
	if( policy == ExecutionPolicy::Parallel_Sequenced || policy == ExecutionPolicy::Parallel_Unsequenced )
		workers = std::max( 1u, std::min( std::thread::hardware_concurrency(), unsigned( rows / 64 + 1 ) ) );
	if( workers == 1 ) { for( Frame r = 0; r < rows; ++r ) body( r ); return; }
	std::vector<std::thread> pool;
	for( unsigned w = 0; w < workers; ++w )
		pool.emplace_back( [=] { for( Frame r = Frame( w ); r < rows; r += Frame( workers ) ) body( r ); } );
	for( auto & t : pool ) t.join();
	}

// The program of an expression Function that is valid, else null after printing why it is not (also null for any other
// Function, silently).
const flan_b200_fx_program * expr_program( const char * what, const Function<TF, float> & f )
	{
	const fx::Expr * e = f.expr();
	if( e && !e->valid() ) std::cout << "flan::" << what << ": " << e->error() << std::endl;
	return e ? e->program() : nullptr;
	}
bool invalid_expr( const char * what, const Function<TF, float> & f ) { return f.expr() && !expr_program( what, f ); }

// What an expression reads decides the view it is sampled into: (B, 1) for t and f, (1, 0) for t, (0, 1) for f, (0, 0)
// for neither.
void expr_view( const flan_b200_fx_program * p, Frame F, Bin B, Frame * rows, Bin * cols, int64_t * frame_stride, int * bin_stride )
	{
	int ut = 0, uf = 0;
	flan_b200_fx_check( p, &ut, &uf );
	*rows = ut ? F : 1; *cols = uf ? B : 1;
	*frame_stride = ut ? *cols : 0; *bin_stride = uf ? 1 : 0;
	}

// sample_function_over_domain (PV.h:31-35): value( frame, bin ) = f( { frame * ( 1 / analysis_rate ), bin * bin_to_frequency( 1 ) } ).
// Host memory; *frame_stride, *bin_stride: (0, 0) for a constant, the expression's view (expr_view) for a valid
// expression, (B, 1) otherwise.
std::vector<float> sample_on_host( const PV & pv, const Function<TF, float> & f, int64_t * frame_stride, int * bin_stride )
	{
	const Frame F = pv.get_num_frames();
	const Bin B = pv.get_num_bins();
	std::vector<float> host;
	*frame_stride = 0; *bin_stride = 0;
	if( f.is_constant() )
		host.assign( 1, f( TF{ 0, 0 } ) );
	else if( const flan_b200_fx_program * p = expr_program( "PV", f ) )
		{
		Frame rows; Bin cols;
		expr_view( p, F, B, &rows, &cols, frame_stride, bin_stride );
		host.resize( size_t( rows ) * size_t( cols ) );
		const float x_scale = 1.0f / pv.get_analysis_rate(), y_scale = pv.bin_to_frequency( 1 );
		for_rows( f.get_execution_policy(), rows, [&]( Frame x )
			{
			for( Bin y = 0; y < cols; ++y ) flan_b200_fx_eval( p, x * x_scale, y * y_scale, &host[size_t( x ) * cols + y] );
			} );
		}
	else
		{
		host.resize( size_t( F ) * size_t( B ) );
		const float x_scale = 1.0f / pv.get_analysis_rate(), y_scale = pv.bin_to_frequency( 1 );
		for_rows( f.get_execution_policy(), F, [&]( Frame x )
			{
			for( Bin y = 0; y < B; ++y ) host[size_t( x ) * B + y] = f( TF{ x * x_scale, y * y_scale } );
			} );
		*frame_stride = B; *bin_stride = 1;
		}
	return host;
	}

int report( flan_b200_ctx * ctx, const char * what, int rc )
	{
	if( rc != FLAN_B200_OK ) std::cout << "flan::" << what << " failed on the GPU engine: " << flan_b200_last_error( ctx ) << std::endl;
	return rc;
	}

// The same table on the device. An expression is sampled there (flan_b200_fx_sample), in its compact view.
bool sample_over_domain( const char * what, const PV & pv, const Function<TF, float> & f, DeviceTable & t )
	{
	if( const flan_b200_fx_program * p = expr_program( what, f ) )
		{
		Frame rows; Bin cols;
		expr_view( p, pv.get_num_frames(), pv.get_num_bins(), &rows, &cols, &t.frame_stride, &t.bin_stride );
		float * d = nullptr;
		t.data = b200::Mirror<float>::device_result( size_t( rows ) * size_t( cols ), &d );
		flan_b200_ctx * ctx = b200::context();
		if( !d || !ctx || report( ctx, what, flan_b200_fx_sample( ctx, p, pv.get_num_frames(), pv.get_num_bins(), 1.0f / pv.get_analysis_rate(),
				pv.bin_to_frequency( 1 ), d, &t.frame_stride, &t.bin_stride ) ) ) return false;
		t.d = d;
		return true;
		}
	t.data = b200::Mirror<float>( sample_on_host( pv, f, &t.frame_stride, &t.bin_stride ) );
	t.d = t.data.device();
	return t.d != nullptr;
	}

int device_interp( const char * what, const Interpolator & interp )
	{
	if( interp.get_device_id() < 0 )
		std::cout << "flan::" << what << ": only the named Interpolators (linear ... sqrt) have a GPU form." << std::endl;
	return interp.get_device_id();
	}

const float * as_floats( const MF * p ) { return reinterpret_cast<const float *>( p ); }

// A PV sharded over several GPUs (Audio::convert_to_PV of a long signal): the multi-device form of repitch, stretch or
// modify_time (include/flan_b200.h) with the host table, and the result stays sharded -- null when the PV is not sharded.
using MultiCall = int ( * )( flan_b200_multi *, const flan_b200_sharded_pv *, const float *, int64_t, int, int, flan_b200_sharded_pv * );
std::optional<PV> on_shards( const PV & me, const char * what, MultiCall call, const Function<TF, float> & f, int interp, bool summaries )
	{
	const auto & store = me.storage().shards();
	flan_b200_multi * m = b200::multi();
	if( !store || !m ) return std::nullopt;
	int64_t fs = 0; int bs = 0;
	const std::vector<float> table = sample_on_host( me, f, &fs, &bs );
	auto out = b200::new_sharded_store();
	auto * desc = static_cast<flan_b200_sharded_pv *>( b200::sharded_descriptor( *out ) );
	if( call( m, static_cast<const flan_b200_sharded_pv *>( b200::sharded_descriptor( *store ) ), table.data(), fs, bs, interp, desc ) != FLAN_B200_OK )
		{
		std::cout << "flan::" << what << " failed on the GPU engine: " << flan_b200_multi_last_error( m ) << std::endl;
		return PV();
		}
	if( summaries ) b200::set_sharded_summaries( *out );
	PVBuffer::Format format = me.get_format();
	format.num_frames = Frame( desc->frames );
	const size_t count = size_t( format.num_channels ) * size_t( format.num_frames ) * size_t( format.num_bins );
	return PV( PVBuffer::from_device_result( format, b200::Mirror<MF>::from_shards( count, std::move( out ) ) ) );
	}

// modify_time_base (PVModify.cpp:307-362) on a device time map in seconds.
PV modify_time_on_device( const PV & me, const char * what, const float * d_map, int64_t fs, int bs, int interp )
	{
	flan_b200_ctx * ctx = b200::context();
	const MF * d_pv = me.storage().device();
	if( !ctx || !d_pv ) return PV();
	int64_t out_frames = 0;
	if( report( ctx, what, flan_b200_modify_time_frames( ctx, d_map, fs, bs, me.get_num_frames(), me.get_num_bins(),
			me.get_sample_rate(), me.get_analysis_rate(), &out_frames ) ) ) return PV();
	PVBuffer::Format format = me.get_format();
	format.num_frames = Frame( std::max<int64_t>( out_frames, 0 ) );      // PVModify.cpp:314-315
	MF * d_out = nullptr;
	b200::Mirror<MF> data = b200::Mirror<MF>::device_result( size_t( format.num_channels ) * size_t( format.num_frames ) * size_t( format.num_bins ), &d_out );
	if( !d_out ) return PV();
	if( report( ctx, what, flan_b200_modify_time( ctx, as_floats( d_pv ), me.get_num_channels(), me.get_num_frames(), me.get_num_bins(),
			me.get_sample_rate(), me.get_analysis_rate(), d_map, fs, bs, interp, out_frames, reinterpret_cast<float *>( d_out ),
			int( me.get_window_size() ) ) ) ) return PV();      // also leaves the phase summaries PV::convert_to_audio needs
	return PV( PVBuffer::from_device_result( format, std::move( data ) ) );
	}

}

PV PV::repitch( const Function<TF, float> & factor, const Interpolator & interp ) const
	{
	if( is_null() ) return PV();                                         // PVModify.cpp:202
	const int id = device_interp( "PV::repitch", interp );
	if( id < 0 || invalid_expr( "PV::repitch", factor ) ) return PV();
	if( auto sharded = on_shards( *this, "PV::repitch", flan_b200_multi_repitch, factor, id, false ) ) return std::move( *sharded );
	flan_b200_ctx * ctx = b200::context();
	DeviceTable t;
	if( id < 0 || !ctx || !sample_over_domain( "PV::repitch", *this, factor, t ) ) return PV();
	const MF * d_pv = storage().device();
	MF * d_out = nullptr;
	b200::Mirror<MF> data = b200::Mirror<MF>::device_result( storage().size(), &d_out );
	if( !d_pv || !d_out ) return PV();
	if( report( ctx, "PV::repitch", flan_b200_repitch( ctx, as_floats( d_pv ), get_num_channels(), get_num_frames(), get_num_bins(),
			get_sample_rate(), t.d, t.frame_stride, t.bin_stride, id, reinterpret_cast<float *>( d_out ) ) ) ) return PV();
	// the factor table dies with this scope: its device block goes back to the engine's cache, which orders the next user
	// after the kernels enqueued here -- no synchronise
	return PV( PVBuffer::from_device_result( get_format(), std::move( data ) ) );
	}

PV PV::modify_frequency( const Function<TF, Frequency> & mod, const Interpolator & interp ) const
	{
	if( is_null() ) return PV();
	const int id = device_interp( "PV::modify_frequency", interp );
	flan_b200_ctx * ctx = b200::context();
	DeviceTable t;
	if( id < 0 || invalid_expr( "PV::modify_frequency", mod ) || !ctx || !sample_over_domain( "PV::modify_frequency", *this, mod, t ) ) return PV();
	const Frame F = get_num_frames(); const Bin B = get_num_bins();
	// mod evaluated at every MF's own frequency (PVModify.cpp:263-268)
	b200::Mirror<float> in_mod;
	const float * d_in_mod = nullptr;
	if( const flan_b200_fx_program * p = expr_program( "PV::modify_frequency", mod ) )
		{
		// an expression: on the device, from the device copy of the PV (frame_to_time( x ) = x / ( sr / hop ))
		const MF * d_src = storage().device();
		float * d = nullptr;
		in_mod = b200::Mirror<float>::device_result( storage().size(), &d );
		if( !d_src || !d || report( ctx, "PV::modify_frequency", flan_b200_fx_at_pv( ctx, p, as_floats( d_src ), get_num_channels(), F, B,
				float( get_sample_rate() ) / float( get_hop_size() ), d ) ) ) return PV();
		d_in_mod = d;
		}
	else
		{
		// a user lambda of the data, so it runs here
		const std::vector<MF> & host = get_buffer();
		std::vector<float> in_modified( host.size() );
		for_rows( mod.get_execution_policy(), Frame( get_num_channels() ) * F, [&]( Frame row )
			{
			const Frame frame = row % F;
			for( Bin bin = 0; bin < B; ++bin )
				in_modified[size_t( row ) * B + bin] = mod( TF{ frame_to_time( frame ), host[size_t( row ) * B + bin].f } );
			} );
		in_mod = b200::Mirror<float>( std::move( in_modified ) );
		d_in_mod = in_mod.device();
		}
	const MF * d_pv = storage().device();
	MF * d_out = nullptr;
	b200::Mirror<MF> data = b200::Mirror<MF>::device_result( storage().size(), &d_out );
	if( !d_in_mod || !d_pv || !d_out ) return PV();
	if( report( ctx, "PV::modify_frequency", flan_b200_modify_frequency( ctx, as_floats( d_pv ), get_num_channels(), F, B, get_sample_rate(),
			t.d, t.frame_stride, t.bin_stride, d_in_mod, id, reinterpret_cast<float *>( d_out ) ) ) ) return PV();
	return PV( PVBuffer::from_device_result( get_format(), std::move( data ) ) );
	}

PV PV::modify_time( const Function<TF, Second> & mod, const Interpolator & interp ) const
	{
	if( is_null() ) return PV();                                         // PVModify.cpp:309
	const int id = device_interp( "PV::modify_time", interp );
	if( id < 0 || invalid_expr( "PV::modify_time", mod ) ) return PV();
	if( auto sharded = on_shards( *this, "PV::modify_time", flan_b200_multi_modify_time, mod, id, true ) ) return std::move( *sharded );
	DeviceTable t;
	if( id < 0 || !b200::context() || !sample_over_domain( "PV::modify_time", *this, mod, t ) ) return PV();
	return modify_time_on_device( *this, "PV::modify_time", t.d, t.frame_stride, t.bin_stride, id );
	}

PV PV::stretch( const Function<TF, float> & factor, const Interpolator & interp ) const
	{
	if( is_null() ) return PV();
	const int id = device_interp( "PV::stretch", interp );
	if( id < 0 || invalid_expr( "PV::stretch", factor ) ) return PV();
	if( auto sharded = on_shards( *this, "PV::stretch", flan_b200_multi_stretch, factor, id, true ) ) return std::move( *sharded );
	flan_b200_ctx * ctx = b200::context();
	DeviceTable t;
	if( id < 0 || !ctx || !sample_over_domain( "PV::stretch", *this, factor, t ) ) return PV();
	// running sum along frames, frames -> seconds (PVModify.cpp:373-382), on the device
	const int cols = t.bin_stride ? get_num_bins() : 1;
	float * d_map = nullptr;
	b200::Mirror<float> map = b200::Mirror<float>::device_result( size_t( get_num_frames() ) * size_t( cols ), &d_map );
	if( !d_map ) return PV();
	if( report( ctx, "PV::stretch", flan_b200_stretch_map( ctx, t.d, t.frame_stride, t.bin_stride, get_num_frames(), get_num_bins(),
			get_sample_rate(), get_analysis_rate(), d_map ) ) ) return PV();
	return modify_time_on_device( *this, "PV::stretch", d_map, cols, t.bin_stride, id );
	}

}
