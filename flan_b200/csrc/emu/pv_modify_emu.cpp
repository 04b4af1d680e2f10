// flan_b200/csrc/emu/pv_modify_emu.cpp -- CPU emulator of the PV-domain kernel bodies in pv_modify_body.cuh.
//
// TEST HARNESS, not a product path (nothing in libflan_b200.so links or calls this): it runs the same per-thread
// phase functions the kernels of pv_modify.cu run, thread by thread between the barriers, with the host-side
// orchestration of pv_capi.cu restated, so that the scatter logic, the monotonicity vote and the chunking can be
// checked against the oracle in a container without a GPU (tests/test_emulator_modify.py). Threads of a phase are run
// in DESCENDING thread order to make any accidental dependence on the order visible.
#include "../pv_modify_body.cuh"

#include <cmath>
#include <cstring>
#include <vector>

using namespace pvm;

namespace {

void repitch_rows( const RepitchArgs & a, int64_t rows, int nt )
	{
	std::vector<unsigned char> smem( RepitchRow::bytes( a.B ) );
	RepitchRow s( smem.data(), a.B );
	for( int64_t row = 0; row < rows; ++row )
		{
		for( int t = nt - 1; t >= 0; --t ) repitch_load( a, row, t, nt, s );
		int flags = 0;
		for( int t = nt - 1; t >= 0; --t ) flags |= repitch_map( a, t, nt, s );
		for( int t = nt - 1; t >= 0; --t ) repitch_scatter( a, flags, t, nt, s );
		for( int t = nt - 1; t >= 0; --t ) repitch_store( a, row, t, nt, s );
		}
	}

bool strides_ok( int64_t fs, int bs, int B ) { return ( bs == 0 || bs == 1 ) && ( fs == 0 || fs == ( bs ? B : 1 ) ); }

int64_t map_frames( const Table & mod, int64_t rows, int cols, float sr, int hop, bool & descends )
	{
	float mx = 0.0f; bool any = false; descends = false;
	for( int64_t i = rows * cols - 1; i >= 0; --i )
		{
		float sec; bool d;
		time_map_check( mod, i / cols, (int)( i % cols ), sec, d );
		if( !any || mx < sec ) mx = sec;
		any = true; descends |= d;
		}
	mx = key_float( float_key( mx ) );
	return (int64_t) to_int( std::ceil( mx * sr / float( hop ) ) );
	}

} // namespace

extern "C" {

int pv_emu_repitch( const float * pv, int C, int64_t F, int B, float sr, const float * factor, int64_t fs, int bs,
                    const float * mod_hz, const float * in_mod, int interp, int threads, float * out )
	{
	if( !strides_ok( fs, bs, B ) ) return 1;
	const int64_t rows = fs ? F : 1;
	std::vector<float> hz( (size_t) rows * B );
	Table mod{ mod_hz, fs, bs };
	if( !mod_hz )
		{
		const Table fac{ factor, fs, bs };
		for( int64_t r = 0; r < rows; ++r ) bin_prefix_row( fac, r, B, sr, float( ( B - 1 ) * 2 ), hz.data() + r * B );
		mod = Table{ hz.data(), fs ? (int64_t) B : 0, 1 };
		}
	RepitchArgs a{};
	a.pv = (const float2 *) pv; a.out = (float2 *) out; a.mod = mod; a.in_mod = in_mod;
	a.F = F; a.B = B; a.bin_width = sr / float( ( B - 1 ) * 2 ); a.interp = interp;
	if( mod.frame_stride == 0 && mod.bin_stride == 1 )
		{
		// plan + gather, as pv_repitch_plan_kernel / pv_repitch_shared_kernel
		std::vector<int> src( B ); std::vector<float> mix( B ), pos( B ); int ok = 0;
		RepitchPlan plan{ src.data(), mix.data(), &ok };
		const int nt = threads;
		for( int t = nt - 1; t >= 0; --t ) repitch_plan_positions( mod.p, B, a.bin_width, t, nt, pos.data(), plan );
		int flags = 0;
		for( int t = nt - 1; t >= 0; --t ) flags |= repitch_plan_flags( B, t, nt, pos.data() );
		for( int t = nt - 1; t >= 0; --t ) repitch_plan_pairs( B, interp, flags, t, nt, pos.data(), plan );
		if( ok )
			{
			std::vector<float> m( B ), fm( B );
			for( int64_t row = 0; row < (int64_t) C * F; ++row )
				{
				for( int b = B - 1; b >= 0; --b )
					{
					const float2 mf = a.pv[row * B + b];
					m[b] = mf.x;
					fm[b] = in_mod ? in_mod[row * B + b] : repitch_lerp( mod.p, B, a.bin_width, mf.y );
					}
				for( int y = B - 1; y >= 0; --y ) a.out[row * B + y] = repitch_gather( y, src.data(), mix.data(), m.data(), fm.data() );
				}
			return 0;
			}
		}
	repitch_rows( a, (int64_t) C * F, threads );
	return 0;
	}

// factor != null: PV::stretch (the map is built first); else map_seconds is the time map of PV::modify_time.
// out == null: returns the output frame count only. force_sequential exercises the reference-order walk.
// n_cuts > 0 (planned form only): the output is computed shard by shard, cut at cuts[0 .. n_cuts] (0, ..., out_frames);
// used_rows (may be null) receives each shard's input row window.
int64_t pv_emu_stretch_sharded( const float * pv, int C, int64_t F, int B, float sr, float ar, const float * factor,
                                const float * map_seconds, int64_t fs, int bs, int interp, int chunk, int force_sequential,
                                int * used_sequential, float * out, const int64_t * cuts, int n_cuts, int64_t * used_rows )
	{
	if( !strides_ok( fs, bs, B ) ) return -1;
	const int hop = (int)( sr / ar );
	const int cols = bs ? B : 1;
	std::vector<float> built;
	Table mod{ map_seconds, fs, bs };
	if( factor )
		{
		built.resize( (size_t) F * cols );
		const Table fac{ factor, fs, bs };
		if( fs == 0 && bs == 0 )
			{
			std::vector<PrefixSeg> segs( PREFIX_MAX_SEGS );
			const int ns = constant_prefix_segments( *factor, F, segs.data() );
			if( ns > PREFIX_MAX_SEGS ) return -2;
			for( int64_t k = F - 1; k >= 0; --k ) built[k] = constant_prefix_value( segs.data(), ns, *factor, k ) / ( sr / float( hop ) );
			}
		else
			{
			std::vector<float> raw( (size_t) F * cols );
			for( int col = 0; col < cols; ++col ) frame_prefix_column( fac, col, F, cols, raw.data() );
			for( int64_t i = F * cols - 1; i >= 0; --i ) frame_prefix_convert( raw.data(), built.data(), i, sr / float( hop ) );
			}
		mod = Table{ built.data(), (int64_t) cols, bs };
		}
	bool descends = false;
	const int64_t out_frames = map_frames( mod, mod.frame_stride ? F : 1, cols, sr, hop, descends );
	if( used_sequential ) *used_sequential = descends || force_sequential;
	if( !out || out_frames <= 0 ) return out_frames;
	StretchArgs a{};
	a.pv = (const float2 *) pv; a.out = (float2 *) out; a.mod = mod;
	a.F = F; a.out_frames = out_frames; a.B = B; a.sample_rate = sr; a.hop = float( hop ); a.interp = interp;
	a.chunk = chunk; a.chunks = ( F - 1 + chunk - 1 ) / chunk;
	if( a.chunks < 1 ) a.chunks = 1;
	a.pv_channel_stride = F * B; a.out_channel_stride = out_frames * B;
	if( !descends && !force_sequential && bs == 0 && n_cuts > 0 )
		{
		// as flan_b200_multi_stretch / _modify_time: the plan of the whole signal, then per output shard
		// [cuts[i], cuts[i+1]) (multiples of seg_len) its row window (stretch_window) staged into a buffer of its own and
		// the shard's segments written into another. Rows outside the window and cells outside the shard are NaN, so a read
		// or write past them changes the result.
		const int seg_len = chunk;
		if( cuts[0] != 0 || cuts[n_cuts] != out_frames ) return -3;
		std::vector<int> xpos( F ); std::vector<float> mix( out_frames ); std::vector<int> src( out_frames, -1 );
		StretchPlan plan{ xpos.data(), mix.data(), src.data() };
		for( int64_t f = F - 1; f >= 0; --f ) stretch_plan_frame( a, plan, f );
		pvk::PvConsts k{};
		const float nan = std::nanf( "" );
		constexpr int64_t GUARD = 2;
		for( int s = n_cuts - 1; s >= 0; --s )
			{
			const int64_t x0 = cuts[s], x1 = cuts[s + 1];
			if( x1 < x0 || x0 % seg_len != 0 ) return -3;
			int64_t r0 = 0, r1 = 0;
			stretch_window( plan, F, x0, x1, &r0, &r1 );
			if( used_rows ) { used_rows[2 * s] = r0; used_rows[2 * s + 1] = r1; }
			const int64_t rows = r1 - r0, in_stride = ( rows + 2 * GUARD ) * B, out_stride = ( x1 - x0 ) * B;
			std::vector<float2> win( (size_t)( C * in_stride ), make_float2( nan, nan ) ), part( (size_t)( C * out_stride ), make_float2( nan, nan ) );
			for( int c = 0; c < C; ++c )
				std::memcpy( win.data() + c * in_stride + GUARD * B, (const float2 *) pv + ( c * F + r0 ) * B, sizeof( float2 ) * rows * B );
			StretchArgs sa = a;
			sa.pv = win.data() + GUARD * B; sa.row0 = r0; sa.pv_channel_stride = in_stride;
			sa.out = part.data(); sa.out_row0 = x0; sa.out_channel_stride = out_stride;
			sa.seg0 = x0 / seg_len;
			const int64_t segs = ( x1 - x0 + seg_len - 1 ) / seg_len;
			for( int c = C - 1; c >= 0; --c )
				for( int64_t sgm = segs - 1; sgm >= 0; --sgm )
					for( int b = B - 1; b >= 0; --b ) stretch_segment_planned<false>( sa, plan, c, sgm, seg_len, b, nullptr, k );
			for( int c = 0; c < C; ++c )
				std::memcpy( (float2 *) out + ( c * out_frames + x0 ) * B, part.data() + c * out_stride, sizeof( float2 ) * out_stride );
			}
		}
	else if( !descends && !force_sequential && bs == 0 )
		{
		// as on the device: plan, then the gather by segments of output frames (`chunk` doubles as the segment length here,
		// so the tests cut segments inside pairs, at pair boundaries and beyond the covered range)
		std::vector<int> xpos( F ); std::vector<float> mix( out_frames ); std::vector<int> src( out_frames, -1 );
		StretchPlan plan{ xpos.data(), mix.data(), src.data() };
		for( int64_t f = F - 1; f >= 0; --f ) stretch_plan_frame( a, plan, f );
		const int seg_len = chunk;
		const int64_t segs = ( out_frames + seg_len - 1 ) / seg_len;
		pvk::PvConsts k{};
		for( int c = C - 1; c >= 0; --c )
			for( int64_t sgm = segs - 1; sgm >= 0; --sgm )
				for( int b = B - 1; b >= 0; --b ) stretch_segment_planned<false>( a, plan, c, sgm, seg_len, b, nullptr, k );
		}
	else if( !descends && !force_sequential )
		{
		for( int c = C - 1; c >= 0; --c )
			for( int64_t k = a.chunks - 1; k >= 0; --k )
				for( int b = B - 1; b >= 0; --b ) stretch_chunk( a, c, k, b );
		}
	else
		{
		std::memset( out, 0, sizeof( float2 ) * (size_t) C * out_frames * B );
		for( int c = 0; c < C; ++c )
			for( int b = 0; b < B; ++b ) stretch_column( a, c, b );
		}
	return out_frames;
	}

int64_t pv_emu_stretch( const float * pv, int C, int64_t F, int B, float sr, float ar, const float * factor,
                        const float * map_seconds, int64_t fs, int bs, int interp, int chunk, int force_sequential,
                        int * used_sequential, float * out )
	{
	return pv_emu_stretch_sharded( pv, C, F, B, sr, ar, factor, map_seconds, fs, bs, interp, chunk, force_sequential,
	                               used_sequential, out, nullptr, 0, nullptr );
	}

}

extern "C" {

// Closed-form running sum of a constant (constant_prefix_segments / constant_prefix_value) against the plain loop:
// returns the number of mismatching elements; *segments receives the segment count.
int64_t pv_emu_constant_prefix_mismatches( float c, int64_t F, int * segments )
	{
	std::vector<PrefixSeg> segs( PREFIX_MAX_SEGS );
	const int ns = constant_prefix_segments( c, F, segs.data() );
	if( segments ) *segments = ns;
	if( ns > PREFIX_MAX_SEGS ) return -1;
	int64_t bad = 0;
	float acc = 0.0f;
	for( int64_t k = 0; k < F; ++k )
		{
		acc = k == 0 ? c : c + acc;
		const float got = constant_prefix_value( segs.data(), ns, c, k );
		if( std::memcmp( &got, &acc, 4 ) != 0 && !( got != got && acc != acc ) ) ++bad;
		}
	return bad;
	}

}
