// flan_b200/csrc/pv_body.cuh
//
// CTA bodies of the analysis (Audio::convert_to_PV, reference Conversions/AudioPV.cpp:12-78) and
// resynthesis (PV::convert_to_audio, AudioPV.cpp:86-139) kernels, written against an Env so that the
// identical source runs on the device (pv_kernels.cu) and in the CPU thread emulator (emu/pv_emu.cpp).
//
// Work decomposition (both directions): a CTA owns one contiguous SEGMENT of frames of one channel and
// walks it in frame order. A frame of N-point real FFT is computed by T = N/16 (8 complex points per thread)
// or N/32 threads (16 points; the real transform is a packed N/2-point complex FFT). Walking in order lets
//   * analysis keep the previous frame's phase of "its" bins in registers (the serial dependency of
//     AudioPV.cpp:47/phase_vocoder.cpp:44-45), at the cost of one warm-up FFT per segment; consecutive
//     windows overlap by W-hop samples, which stay in L1, so each input sample leaves HBM once;
//   * resynthesis keep the fp64 phase accumulators (phase_vocoder.cpp:58-59) in registers and the
//     overlap-add in a shared-memory ring, so every output sample is written once, contributions added in
//     increasing frame order like AudioPV.cpp:133-134.
// Window coefficients and bin constants for a thread's fixed positions stay in registers across the walk;
// every shared-memory access is "per-thread base + immediate" (see xpad in pv_core.cuh).
//
// Bodies: analysis_cta (8 / 16 points per thread, any window and hop), analysis_cta_mirror and
// synthesis_cta_mirror (16 points, the butterfly pair (p, NS-p) in one thread: window == dft, hop == dft/16),
// synthesis_cta (8 points, any window and hop). DESIGN.md section 4 says which one serves which call and why.
#pragma once

#include "pv_core.cuh"

namespace pvk {

// ------------------------------------------------------------------------------------------------
// FFT pass chain over the ping-pong exchange buffers x0/x1 (XBuf<M>::size float2 each).
// Pass 0 (radix 8 or 16, no twiddles) is issued by the caller; this runs passes 1..last.
// ------------------------------------------------------------------------------------------------
// Twiddles of pass p into w[] (at most PT-1 values); no-op past the last pass.
template<int M, int PT, int p, class Env>
PV_HD void fft_chain_twiddles( int t, float2 * w, const float2 * tw, Env & env )
	{
	using P = FftPlan<M, PT>;
	if constexpr( p < P::num_passes )
		fft_load_twiddles<M, PT, P::radix( p ), P::ns( p )>( t, w, tw + P::tw_offset( p ), [&]( const float2 * q ) { return env.ldg2( q ); } );
	}

// PRE: `w` holds the twiddles of pass p on entry: the caller requests them (fft_chain_twiddles) BEFORE the barrier that
// publishes pass p-1's outputs, and each pass requests the next one's before its own barrier, so the table reads never
// wait behind a barrier. Measured: a gain where registers are free at the barrier (resynthesis), a loss in the
// analysis kernels, whose 128 registers are full (cfg2 1.66 -> 1.70 ms); those read the table inside the pass (!PRE).
template<int M, int PT, int p, bool STORE_LAST, bool ONE, bool PRE, class Env>
PV_HD void fft_pass_chain( int t, float2 * v, float2 * x0, float2 * x1, const float2 * tw, Env & env, float2 * w )
	{
	using P = FftPlan<M, PT>;
	if constexpr( p < P::num_passes )
		{
		constexpr int NSp = P::ns( p - 1 );     // layout our input was written in
		constexpr int R = P::radix( p ), NS = P::ns( p );
		// ONE: a single exchange buffer (half the shared memory, so more L1 for the tables, and one base register less)
		// at the price of a barrier between a pass's reads and its writes
		float2 * in  = ( ONE || ( p - 1 ) % 2 == 0 ) ? x0 : x1;
		float2 * out = ( ONE || p % 2 == 0 ) ? x0 : x1;
		fft_load<M, PT, NSp>( t, v, in );
		// everyone has read before anyone writes (a last pass that stores nothing needs no such barrier)
		if constexpr( ONE && ( p < P::num_passes - 1 || STORE_LAST ) ) env.sync();
		if constexpr( PRE ) fft_butterflies_w<M, PT, R, NS>( v, w );
		else fft_butterflies<M, PT, R, NS>( t, v, tw + P::tw_offset( p ), [&]( const float2 * q ) { return env.ldg2( q ); } );
		if constexpr( p < P::num_passes - 1 )
			{
			fft_store<M, PT, R, NS>( t, v, out );
			if constexpr( PRE ) fft_chain_twiddles<M, PT, p + 1>( t, w, tw, env );
			env.sync();
			}
		else if constexpr( STORE_LAST )
			{
			// Last pass: its outputs are in natural order, v[s] = Z[t + s*T]. The real-FFT unpack pairs Z[k] with
			// Z[M-k]: the lower half (s < PT/2) stays in this thread's registers, only the upper half is published.
#pragma unroll
			for( int s = PT / 2; s < PT; ++s ) out[t + s * ( M / PT )] = v[s];
			env.sync();
			}
		fft_pass_chain<M, PT, p + 1, STORE_LAST, ONE, PRE>( t, v, x0, x1, tw, env, w );
		}
	}

// Buffer that receives the natural-order output of the last pass when STORE_LAST is set (its Ns >= 16: no padding).
template<int M, int PT, bool ONE = false> PV_HD float2 * fft_result_buffer( float2 * x0, float2 * x1 )
	{
	return ( ONE || ( FftPlan<M, PT>::num_passes - 1 ) % 2 == 0 ) ? x0 : x1;
	}

// ------------------------------------------------------------------------------------------------
// Analysis
// ------------------------------------------------------------------------------------------------
struct AnalysisArgs
	{
	const float * audio;        // local buffer; channel c starts at audio + c * audio_stride
	int64_t audio_stride;       // elements between channels of the local buffer
	int64_t audio_offset;       // absolute sample index held at local position 0 (frame-range shards)
	int64_t n_total;            // samples per channel of the whole signal; reads outside [0,n_total) are 0
	float2 * pv;                // rows of (m,f): pv + c * pv_channel_stride + (frame - frame_begin) * B
	int64_t pv_channel_stride;
	int64_t frame_begin, frame_end;   // absolute frames produced by this launch
	int seg_len;                // frames per CTA
	int segs_per_channel;
	int W, hop;
	int aligned2;               // every in-signal window of every channel starts on an 8-byte boundary
	const float * win;          // [W] Hann, reference expression evaluated on the host
	const float2 * binc;        // [B] (bin_to_frequency(b), expected_phase_diff(b)), host-evaluated
	                            //     (PVBuffer.cpp:443-446, phase_vocoder.cpp:47)
	const float4 * binc4;       // [N/4+1] the same constants per unpack pair: (binf[k], binf[M-k], expected[k], -expected[M-k])
	const float2 * post_rot;    // [N/4+1] -i e^{-2 pi i k/N}
	const float2 * pass_tw;     // concatenated per-pass twiddles
	int one_buffer;             // the two exchange buffers alias (half the shared memory, two more barriers per frame)
	PvConsts k;
	// EMIT instantiations only: the phase summaries PV::convert_to_audio needs of the rows this launch writes
	// ([C][segs_per_channel][B], the layout of pv_phase_seg_kernel's output; entries the fast form cannot produce carry a
	// NaN in sum.q and are recomputed from the rows by the scan), P = double( pi2 ), rcpP = 1 / P
	PhaseSeg * seg_out;
	double P, rcpP;
	};

// Tensor memory of the 16-point analysis at dft 4096 (128 threads: thread t owns TMEM lane t; 128 columns per CTA, so the
// four CTAs an SM holds at 128 registers use all 512 columns). What a thread reads every frame and never changes during
// the walk is stored there once, instead of living in registers (the window) or being re-read through L1 (the tables):
//   columns  0..31  window coefficients w[0..31]
//           32..59  the 14 twiddles of the last pass (radix 8, two butterflies)
//           60      EMIT: the sum of bin M/2 (thread T/2; the other threads' column 60 stays zero)
//           64..127 per slot u, 8 columns: binc4[k] (4), post_rot[k] (2), EMIT: the sums of bins k and M-k (2), k = t + u*T
// The first pass's twiddles stay in L1: their index is t mod 16, 240 entries in all. The sums (EMIT, below) are int32
// bit patterns; they start as the zeros the table stores write.
template<int N, int PT> constexpr bool analysis_tmem() { return PT == 16 && N == 4096; }
constexpr int AN_TM_COLS = 128, AN_TM_WIN = 0, AN_TM_TW = 32, AN_TM_MID = 60, AN_TM_BIN = 64, AN_TM_SUM = 6;

// PAD: a zero-padded window that fills whole slots of the thread layout (window a multiple of 2T samples, < dft: the
// API default window 2048 / dft 4096, Audio.h:158-163) loads its samples as vectors like the full window does; a
// separate instantiation so that the full-window kernels keep their register budget.
// EMIT: the CTA also leaves the phase summary of its segment (DESIGN.md 4.2) -- what pv_phase_seg_kernel would compute
// from a second read of the rows. A bin's increment inc = float( f / ar * pi2 ) lies within pi of its expected phase
// advance c (the table value the phase vocoder subtracts); from c >= 2 and inc >= 2 on both are multiples of 2^-22, so
// d = inc - c is exact, |d| < 4, and the segment's sum of up to 128 such d fits an int32 in units of 2^-22: ONE shared-
// memory word per bin, private to the thread that owns the bin (`ssum`, M + 1 ints; TM: two spare columns of the slot's
// group of the tensor-memory layout and column AN_TM_MID, read with the slot's constants), no registers. The total
// frames * c + 2^-22 * sum is exact in double and equals the plain double running sum of pv_phase_seg_kernel bit for
// bit (that sum is exact too: multiples of 2^-22 below 2^18); increments are positive, so the running maximum is the
// total. A bin that ever leaves those conditions (the lowest bins, NaN / Inf) is marked and gets the NaN entry.
// TM: the tensor-memory form (analysis_tmem); the Env then addresses the CTA's AN_TM_COLS columns.
template<int N, int PT, bool ONE, bool PAD, bool EMIT = false, bool TM = analysis_tmem<N, PT>(), class Env>
PV_HD void analysis_cta( const AnalysisArgs & a, int64_t block, Env & env, float2 * x0, float2 * x1, int * ssum = nullptr )
	{
	constexpr int M = N / 2, T = M / PT, H = PT / 2;      // H pairs of bins (k, M-k) per thread
	using P = FftPlan<M, PT>;
	static_assert( !TM || ( T == 128 && P::num_passes == 3 && 2 * PT == 32 && ( P::radix( 2 ) - 1 ) * ( PT / P::radix( 2 ) ) == 14 && H * 8 == 64 ),
	               "tensor-memory layout of the dft-4096 analysis" );
	const int t = env.tid;
	const int c = (int)( block / a.segs_per_channel );
	const int seg = (int)( block % a.segs_per_channel );
	const int64_t fa = a.frame_begin + (int64_t) seg * a.seg_len;
	const int64_t fb = ( fa + a.seg_len < a.frame_end ) ? fa + a.seg_len : a.frame_end;
	if( fa >= fb ) return;

	const float * xch = a.audio + (int64_t) c * a.audio_stride;
	const int W = a.W, hop = a.hop;
	const int half = W / 2;

	// Per-thread constants for its fixed window positions and bins. The window carries a factor 1/2 (exact) that
	// the real-FFT unpack would otherwise apply per bin: 0.5*(x*w) == x*(0.5*w) bit for bit.
	float w[2 * PT];
#pragma unroll
	for( int s = 0; s < PT; ++s )
		{
		const int i0 = 2 * ( t + s * T );
		w[2 * s]     = ( i0 < W )     ? 0.5f * env.ldg( a.win + i0 ) : 0.0f;
		w[2 * s + 1] = ( i0 + 1 < W ) ? 0.5f * env.ldg( a.win + i0 + 1 ) : 0.0f;
		}
	if constexpr( TM )
		{
		env.template tmem_st<32>( AN_TM_WIN, w );
		float2 tw2[16];
		fft_load_twiddles<M, PT, P::radix( 2 ), P::ns( 2 )>( t, tw2, a.pass_tw + P::tw_offset( 2 ), [&]( const float2 * q ) { return env.ldg2( q ); } );
		tw2[14].x = tw2[14].y = tw2[15].x = tw2[15].y = 0.0f;
		env.template tmem_st<32>( AN_TM_TW, reinterpret_cast<const float *>( tw2 ) );
#pragma unroll
		for( int h = 0; h < 2; ++h )
			{
			float tb[32];
#pragma unroll
			for( int j = 0; j < 4; ++j )
				{
				const int k = t + ( 4 * h + j ) * T;
				const float4 cc = env.ldg4( a.binc4 + k );
				const float2 pr = env.ldg2( a.post_rot + k );
				tb[8 * j] = cc.x; tb[8 * j + 1] = cc.y; tb[8 * j + 2] = cc.z; tb[8 * j + 3] = cc.w;
				tb[8 * j + 4] = pr.x; tb[8 * j + 5] = pr.y; tb[8 * j + 6] = 0.0f; tb[8 * j + 7] = 0.0f;
				}
			env.template tmem_st<32>( AN_TM_BIN + 32 * h, tb );
			}
		env.tmem_wait_st();
		env.template tmem_ld<32>( AN_TM_WIN, w );           // the first frame's window; every later one is requested a frame ahead
		}
	// Bins of this thread: slot u holds k = t + u*T and its mirror M-k (k = 0: DC and Nyquist), whose previous phases
	// travel as one packed pair; bin M/2 is the extra bin of thread T/2.
	float2 prev[H];
	float prev_mid = 0.0f;
#pragma unroll
	for( int u = 0; u < H; ++u ) { prev[u].x = 0.0f; prev[u].y = 0.0f; }

	unsigned dirty = 0;             // EMIT: bit 2u / 2u+1 = bin k / M-k of slot u left the fast form, bit 2H = bin M/2
	if( EMIT )
		{
#pragma unroll
		for( int u = 0; u < H; ++u )
			{
			if( !TM ) { ssum[t + u * T] = 0; ssum[M - t - u * T] = 0; }
			const float4 cc = env.ldg4( a.binc4 + ( t + u * T ) );
			dirty |= ( cc.z >= 6.0f ? 0u : 1u << ( 2 * u ) ) | ( -cc.w >= 6.0f ? 0u : 2u << ( 2 * u ) );
			}
		if( t == T / 2 ) { if( !TM ) ssum[M / 2] = 0; dirty |= env.ldg2( a.binc + M / 2 ).y >= 6.0f ? 0u : 1u << ( 2 * H ); }
		}
	// EMIT, TM: the warp of thread T/2 reads and writes column AN_TM_MID together (tcgen05 is warp-wide)
	const bool mid_warp = ( t >> 5 ) == ( ( T / 2 ) >> 5 );

	// The serial reference loop carries frame f-1's phase into frame f (phase_vocoder.cpp:44-45); a segment
	// that does not start at frame 0 recomputes it with one warm-up FFT.
	const int64_t first = ( fa > 0 ) ? fa - 1 : fa;
	// PAD: slots s < slots_in hold sample pairs, the rest of the transform's input is the zero padding of AudioPV.cpp:65
	const bool full_window = ( PAD ? ( W % ( 2 * T ) == 0 ) : ( W == N ) ) && a.aligned2;
	const int slots_in = PAD ? W / ( 2 * T ) : PT;

	// Output row of frame f: bins k = t + u*T ascend from row_lo, their mirrors M-k descend from row_hi (per-thread
	// bases advanced by one row per frame, so every store address is base + immediate). The warm-up frame's row lies
	// before the first one and is never dereferenced.
	const int64_t row0 = (int64_t) c * a.pv_channel_stride + ( first - a.frame_begin ) * (int64_t)( M + 1 );
	float2 * row_lo = a.pv + ( row0 + t );
	float2 * row_hi = a.pv + ( row0 + M - t );
	float2 * row_mid = a.pv + ( row0 + M / 2 );

	for( int64_t f = first; f < fb; ++f, row_lo += M + 1, row_hi += M + 1, row_mid += M + 1 )
		{
		const int64_t start = (int64_t) hop * f - half;                 // AudioPV.cpp:52
		const float * src = xch + ( start - a.audio_offset ) + 2 * t;   // this thread's first sample pair
		float2 v[PT];
		if constexpr( TM ) env.template tmem_wait<2 * PT>( w );
		// pass 0: windowed load (AudioPV.cpp:54-62; zero padding :65) + radix-PT. Windows overlap by W-hop samples:
		// all but the newest hop are L1 hits.
		if( !PAD && full_window && start >= 0 && start + W <= a.n_total )
			{
#pragma unroll
			for( int s = 0; s < PT; ++s )
				{
				const float2 r = env.ldg2( reinterpret_cast<const float2 *>( src + 2 * s * T ) );
				float2 ww; ww.x = w[2 * s]; ww.y = w[2 * s + 1];
				v[s] = mul2( r, ww );
				}
			}
		else if( PAD && full_window && start >= 0 && start + W <= a.n_total )
			{
			// zero-padded window: the same vector loads for the slots that hold samples
#pragma unroll
			for( int s = 0; s < PT; ++s )
				{
				float2 r; r.x = 0.0f; r.y = 0.0f;
				if( s < slots_in ) r = env.ldg2( reinterpret_cast<const float2 *>( src + 2 * s * T ) );
				float2 ww; ww.x = w[2 * s]; ww.y = w[2 * s + 1];
				v[s] = mul2( r, ww );
				}
			}
		else
			{
#pragma unroll
			for( int s = 0; s < PT; ++s )
				{
				const int i0 = 2 * ( t + s * T );
				const int64_t p0 = start + i0, p1 = p0 + 1;
				const float r0 = ( i0 < W && p0 >= 0 && p0 < a.n_total )     ? env.ldg( src + 2 * s * T ) : 0.0f;
				const float r1 = ( i0 + 1 < W && p1 >= 0 && p1 < a.n_total ) ? env.ldg( src + 2 * s * T + 1 ) : 0.0f;
				v[s].x = mul_rn( r0, w[2 * s] );
				v[s].y = mul_rn( r1, w[2 * s + 1] );
				}
			}
		fft_butterflies<M, PT, PT, 1>( t, v, (const float2 *) nullptr, [&]( const float2 * q ) { return env.ldg2( q ); } );
		fft_store<M, PT, PT, 1>( t, v, x0 );
		env.sync();

		// pull the next frame's newest samples towards L1 while this frame computes
		if( f + 1 < fb )
			{
			const int64_t p = start + W + (int64_t) t * 32;
			if( t * 32 < hop && p >= 0 && p < a.n_total ) env.prefetch( xch + ( p - a.audio_offset ) );
			}

		float tab[2][8];            // TM: binc4[k] and post_rot[k] of slot u in tab[u & 1]
		if constexpr( TM )
			{
			// the fft_pass_chain of passes 1 and 2 with the last pass's twiddles from tensor memory, requested before the
			// barrier that publishes the pass's inputs (as are the first slot's bin constants before the unpack's barrier)
			float2 * x = ONE ? x0 : x1;
			fft_load<M, PT, 1>( t, v, x0 );
			if constexpr( ONE ) env.sync();
			fft_butterflies<M, PT, PT, P::ns( 1 )>( t, v, a.pass_tw + P::tw_offset( 1 ), [&]( const float2 * q ) { return env.ldg2( q ); } );
			fft_store<M, PT, PT, P::ns( 1 )>( t, v, x );
			float2 tw2[14];
			env.template tmem_ld<16>( AN_TM_TW, reinterpret_cast<float *>( tw2 ) );
			env.template tmem_ld<8>( AN_TM_TW + 16, reinterpret_cast<float *>( tw2 ) + 16 );
			env.template tmem_ld<4>( AN_TM_TW + 24, reinterpret_cast<float *>( tw2 ) + 24 );
			env.sync();
			fft_load<M, PT, P::ns( 1 )>( t, v, x );
			if constexpr( ONE ) env.sync();
			env.template tmem_wait<28>( reinterpret_cast<float *>( tw2 ) );
			fft_butterflies_w<M, PT, P::radix( 2 ), P::ns( 2 )>( v, tw2 );
			if constexpr( EMIT ) env.tmem_wait_st();       // the sums the previous frame stored (long done) are read next
			env.template tmem_ld<8>( AN_TM_BIN, tab[0] );
#pragma unroll
			for( int s = PT / 2; s < PT; ++s ) x0[t + s * T] = v[s];
			env.sync();
			}
		else
			{
#ifndef PV_ABL_NOFFT
			fft_pass_chain<M, PT, 1, true, ONE, false>( t, v, x0, x1, a.pass_tw, env, (float2 *) nullptr );
#endif
			}
		const float2 * z = fft_result_buffer<M, PT, ONE>( x0, x1 );     // upper half of Z/2 in natural order

		// real-FFT unpack + phase vocoder (AudioPV.cpp:69-73). The warm-up frame runs the same code with its stores
		// predicated off: only the phases it leaves in prev[] matter.
		const bool emit = ( f >= fa );
		float mid[2];               // EMIT, TM: columns AN_TM_MID, +1 of the warp of thread T/2, requested with slot H-1's constants
#pragma unroll
		for( int u = 0; u < H; ++u )
			{
			const float * tu = tab[u & 1];
			const int k = t + u * T;
			// X[k] = (Zk + conj Zm) + (-i w_k)(Zk - conj Zm),  conj X[M-k] = (Zk + conj Zm) - (-i w_k)(Zk - conj Zm), Zm = Z[M-k].
			// k = 0 pairs Z[0] with itself and yields DC in X[k] and Nyquist (bin M) in X[M-k], both real.
			const float2 zk = v[u];
			float2 zm = z[( u == 0 && t == 0 ) ? M / 2 : M - k];
			if( u == 0 && t == 0 ) zm = v[0];
			const float2 A = add2( zk, pn2( zm ) );
			const float2 D = add2( zk, np2( zm ) );
#ifndef PV_ABL_NOTAB
			float2 rot;
			float4 cc;
			if constexpr( TM )
				{
				// slot u's constants (and sums) were requested one slot ahead (slot 0's before the barrier)
				env.template tmem_wait<EMIT ? 8 : 6>( tab[u & 1] );
				if( EMIT && u == H - 1 && emit && mid_warp ) env.template tmem_wait<2>( mid );
				cc.x = tu[0]; cc.y = tu[1]; cc.z = tu[2]; cc.w = tu[3]; rot.x = tu[4]; rot.y = tu[5];
				if( u + 1 < H ) env.template tmem_ld<8>( AN_TM_BIN + 8 * ( u + 1 ), tab[( u + 1 ) & 1] );
				if( EMIT && u + 1 == H - 1 && emit && mid_warp ) env.template tmem_ld<2>( AN_TM_MID, mid );
				}
			else
				{
				rot = env.ldg2( a.post_rot + k );
				cc = env.ldg4( a.binc4 + k );
				}
			const float2 Pq = cmul2( D, rot );
			const float2 xk = add2( A, Pq ), xmc = sub2( A, Pq );
#else
			float2 wq; wq.x = 0.5f + k; wq.y = 0.25f;                        // ablation build only: no table traffic
			const float2 Pq = cmul2( D, wq );
			const float2 xk = add2( A, Pq ), xmc = sub2( A, Pq );
			float4 cc; cc.x = k; cc.y = M - k; cc.z = 0.1f * k; cc.w = -0.1f * k;
#endif
			float2 binf, expd; binf.x = cc.x; binf.y = cc.y; expd.x = cc.z; expd.y = cc.w;
			float2 mk, mm;
#ifndef PV_ABL_NOEPI
			phase_vocoder_pair( xk, xmc, prev[u], binf, expd, a.k, mk, mm );
#else
			mk = add2( xk, binf ); mm = add2( xmc, expd );               // ablation build only
#endif
			if( emit )
				{
				env.st_stream2( row_lo + u * T, mk );
				env.st_stream2( row_hi - u * T, mm );
				if( EMIT )
					{
					// both bins at once; a bin whose expected advance is below 6 rad was marked before the walk, for the others
					// |d| < 4 implies inc > 2 (a NaN fails the comparison); sums of marked bins are never read
					float2 Fq; Fq.x = mk.y; Fq.y = mm.y;
					// phase_increment of both bins. The product is rounded on its own (scalar __fmul_rn): nvcc contracts the packed
					// multiply with the packed subtraction that follows into one FFMA2, i.e. inc * pi2 - c with a single rounding.
					const float2 qq = div_const2( Fq, a.k.analysis_rate, a.k.rcp_analysis_rate );
					float2 inc; inc.x = mul_rn( qq.x, a.k.pi2 ); inc.y = mul_rn( qq.y, a.k.pi2 );
					float2 cen; cen.x = expd.x; cen.y = -expd.y;
					float2 dd; dd.x = sub_rn( inc.x, cen.x ); dd.y = sub_rn( inc.y, cen.y );
					const float2 sc = mul2( dd, splat2( 4194304.0f ) );                     // (inc - c) * 2^22: exact, an integer
					const bool ok_k = fabsf( sc.x ) < 16777216.0f && fabsf( mk.x ) <= 3.402823466e38f;
					const bool ok_m = fabsf( sc.y ) < 16777216.0f && fabsf( mm.x ) <= 3.402823466e38f;
					if constexpr( TM )
						{
						float s2[2];
						s2[0] = int_bits_add( tu[AN_TM_SUM], (int) sc.x );
						s2[1] = int_bits_add( tu[AN_TM_SUM + 1], (int) sc.y );
						env.template tmem_st<2>( AN_TM_BIN + 8 * u + AN_TM_SUM, s2 );
						}
					else
						{
						env.shared_add( ssum + k, (int) sc.x );
						env.shared_add( ssum + ( M - k ), (int) sc.y );
						}
					dirty |= ( ok_k ? 0u : 1u << ( 2 * u ) ) | ( ok_m ? 0u : 2u << ( 2 * u ) );
					}
				}
			}
		if constexpr( TM ) { if( f + 1 < fb ) env.template tmem_ld<2 * PT>( AN_TM_WIN, w ); }     // the next frame's window
		int mid_add = 0;            // EMIT, TM: what thread T/2 adds to its column AN_TM_MID (the rest of its warp adds 0)
		if( t == T / 2 )
			{
			const float2 zh = z[M / 2];                           // X[M/2] = conj(Z[M/2])
			const float2 ch = env.ldg2( a.binc + M / 2 );
			const float2 mh = phase_vocoder_bin( 2.0f * zh.x, -2.0f * zh.y, prev_mid, ch.x, ch.y, a.k );
			if( emit ) env.st_stream2( row_mid, mh );
			if( EMIT && emit )
				{
				const float sc = mul_rn( sub_rn( phase_increment( mh.y, a.k ), ch.y ), 4194304.0f );
				const bool ok = fabsf( sc ) < 16777216.0f && fabsf( mh.x ) <= 3.402823466e38f;
				if( TM ) mid_add = (int) sc;
				else env.shared_add( ssum + M / 2, (int) sc );
				dirty |= ok ? 0u : 1u << ( 2 * H );
				}
			}
		if constexpr( EMIT && TM )
			{
			if( emit && mid_warp )
				{
				mid[0] = int_bits_add( mid[0], mid_add );
				env.template tmem_st<2>( AN_TM_MID, mid );
				}
			}
		// the next frame's pass 0 writes x0, last read two barriers ago; its pass 1 writes x1 after one more barrier
		if( ONE || ( FftPlan<M, PT>::num_passes - 1 ) % 2 == 0 ) env.sync();
		}
	if( EMIT )
		{
		PhaseSeg * out = a.seg_out + ( (int64_t) c * a.segs_per_channel + seg ) * (int64_t)( M + 1 );
		const double frames = (double)( fb - fa );
		auto put = [&]( int bin, float center, bool bad, int sum )
			{
			PhaseSeg s;
			const double total = frames * (double) center + (double) sum * 2.384185791015625e-07;    // 2^-22; exact
			phase_sum_from_double( total, a.P, a.rcpP, s.sum.q, s.sum.r );
			s.mx = s.sum;                                                 // every increment was positive
			if( bad ) s.sum.q = nan_marker();
			out[bin] = s;
			};
		if constexpr( TM ) env.tmem_wait_st();
#pragma unroll
		for( int u = 0; u < H; ++u )
			{
			const int k = t + u * T;
			int sk, sm;
			if constexpr( TM )
				{
				float s2[2];
				env.template tmem_ld<2>( AN_TM_BIN + 8 * u + AN_TM_SUM, s2 );
				env.template tmem_wait<2>( s2 );
				sk = int_bits( s2[0] ); sm = int_bits( s2[1] );
				}
			else { sk = ssum[k]; sm = ssum[M - k]; }
			const float4 cc = env.ldg4( a.binc4 + k );
			put( k, cc.z, ( dirty >> ( 2 * u ) ) & 1u, sk );
			put( M - k, -cc.w, ( dirty >> ( 2 * u + 1 ) ) & 1u, sm );           // slot (0, 0): DC in lane x, Nyquist (bin M) in lane y
			}
		int smid = 0;
		if constexpr( TM )
			{
			if( mid_warp )
				{
				float s2[2];
				env.template tmem_ld<2>( AN_TM_MID, s2 );
				env.template tmem_wait<2>( s2 );
				smid = int_bits( s2[0] );
				}
			}
		else if( t == T / 2 ) smid = ssum[M / 2];
		if( t == T / 2 ) put( M / 2, env.ldg2( a.binc + M / 2 ).y, ( dirty >> ( 2 * H ) ) & 1u, smid );
		}
	}

// ------------------------------------------------------------------------------------------------
// Analysis, mirrored last pass (16 points per thread, dft 1024 / 2048 / 4096: passes 16, 16, R with R = 2 / 4 / 8)
//
// The last Stockham pass consists of NS = M/R butterflies; butterfly j produces Z[j + r*NS], r = 0..R-1, and the
// real-FFT unpack pairs Z[k] with Z[M-k] = Z[(NS-j) + (R-1-r)*NS], i.e. butterfly j with butterfly NS-j. Here one
// thread computes BOTH butterflies of such a pair (p, NS-p), p = t + q*T, so the unpack and the phase vocoder run
// entirely on the thread's own registers: no third exchange through shared memory, no barrier after the last pass.
// The one irregular pair is p = 0: butterflies 0 and NS/2 are each their own mirror (thread 0, q = 0); that thread
// publishes its 2R values and 2R+1 lanes of its warp finish the bins that are multiples of NS/2 one each.
// Samples: a thread's window positions are the same absolute samples in every frame (window == dft, hop == dft/16),
// so it keeps them in a private ring in shared memory and fetches one new pair per frame, one frame ahead.
// Same butterflies and per-bin operation order as analysis_cta; bins above M/2 of the upper slots are computed as
// X[k] directly instead of through the conjugate of their mirror, so results agree to rounding (parity-tested alike).
// ------------------------------------------------------------------------------------------------
template<int R, int S> PV_HD void dft_r( float2 * a )
	{
	if( R == 16 ) dft16<S>( a );
	if( R == 8 ) dft8<S>( a );
	if( R == 4 ) dft4<S>( a );
	if( R == 2 ) dft2<S>( a );
	}

template<int N> struct MirrorPlan
	{
	static constexpr int PT = 16, M = N / 2, T = M / PT;
	using P = FftPlan<M, PT>;                    // the analysis kernel's passes 16, 16, R (dft 1024 / 2048 / 4096)
	static constexpr int R = ( M >= 2048 ) ? 8 : M / 256;    // radix of the mirrored pass: 2, 4, 8 (dft 8192: 8, resynthesis only)
	static constexpr int NS = M / R;             // its butterfly count (256; 512 at dft 8192)
	static constexpr int Q = PT / R / 2;         // mirrored butterfly pairs per thread
	static constexpr int KHI = -( M - NS ) / 2;  // bin offset of the upper slots of the irregular pair
	};

template<int N, class Env>
PV_HD void analysis_cta_mirror( const AnalysisArgs & a, int64_t block, Env & env, float2 * x0, float2 * x1, float2 * ring, float2 * scratch )
	{
	using MP = MirrorPlan<N>;
	using P = typename MP::P;
	static_assert( P::num_passes == 3 && P::last_r == MP::R, "mirrored analysis needs radices 16, 16, R" );
	constexpr int PT = 16, M = MP::M, T = MP::T, R = MP::R, NS = MP::NS, Q = MP::Q;
	constexpr int hop = 2 * T, half = N / 2;           // window == N, hop == N/16 (checked by the launcher)
	const int t = env.tid;
	const int c = (int)( block / a.segs_per_channel );
	const int seg = (int)( block % a.segs_per_channel );
	const int64_t fa = a.frame_begin + (int64_t) seg * a.seg_len;
	const int64_t fb = ( fa + a.seg_len < a.frame_end ) ? fa + a.seg_len : a.frame_end;
	if( fa >= fb ) return;

	const float * xch = a.audio + (int64_t) c * a.audio_stride;

	float w[2 * PT];
#pragma unroll
	for( int s = 0; s < PT; ++s )
		{
		w[2 * s]     = 0.5f * env.ldg( a.win + 2 * ( t + s * T ) );
		w[2 * s + 1] = 0.5f * env.ldg( a.win + 2 * ( t + s * T ) + 1 );
		}
	float2 prev[Q][R];
	float prev_irr = 0.0f;
#pragma unroll
	for( int q = 0; q < Q; ++q )
#pragma unroll
		for( int r = 0; r < R; ++r ) { prev[q][r].x = 0.0f; prev[q][r].y = 0.0f; }

	const int64_t first = ( fa > 0 ) ? fa - 1 : fa;
	const bool irregular = ( t == 0 );                 // owner of the butterflies 0 and NS/2
	const bool warp0 = ( t < 32 );

	// The window of frame f is sample pairs t + T*(f + s - 8), s = 0..15, of this thread: the same absolute samples
	// reappear one slot lower in the next frame, so each thread keeps ITS 16 pairs in a private ring (entry
	// (f + s + 8) & 15 at ring[t + T*entry], i.e. the natural circular buffer of N samples) and fetches ONE new pair
	// per frame, a frame ahead. Samples outside [0, n_total) read as zero (AudioPV.cpp:54-62).
	auto load_pair = [&]( int64_t f, int s )
		{
		const int64_t pos = (int64_t) hop * f - half + 2 * ( t + s * T );
		const float * src = xch + ( pos - a.audio_offset );
		float2 r; r.x = 0.0f; r.y = 0.0f;
		if( f < fb )        // frames past the segment are never transformed, and their samples may lie outside the local buffer
			{
			if( a.aligned2 && pos >= 0 && pos + 1 < a.n_total ) r = env.ldg2( reinterpret_cast<const float2 *>( src ) );
			else
				{
				if( pos >= 0 && pos < a.n_total ) r.x = env.ldg( src );
				if( pos + 1 >= 0 && pos + 1 < a.n_total ) r.y = env.ldg( src + 1 );
				}
			}
		return r;
		};
#pragma unroll 1
	for( int s = 0; s < PT; ++s ) ring[t + T * (int)( ( first + s + 8 ) & 15 )] = load_pair( first, s );
	float2 nxt = load_pair( first + 1, PT - 1 );        // beyond the last frame this reads zeros or real samples; never used

	// Output row of frame f; per-thread bases advanced by one row per frame.
	const int64_t row0 = (int64_t) c * a.pv_channel_stride + ( first - a.frame_begin ) * (int64_t)( M + 1 );
	float2 * row_lo = a.pv + ( row0 + t );             // bins k = p + r*NS ascend from here
	float2 * row_hi = a.pv + ( row0 + M - t );         // mirrors M-k descend from here
	float2 * row_irr = a.pv + ( row0 + ( NS / 2 ) * ( t & 31 ) );   // lanes 0..2R of warp 0: bin (NS/2)*lane
	const float2 * tw_last = a.pass_tw + P::tw_offset( 2 );
	auto ldtw = [&]( const float2 * q ) { return env.ldg2( q ); };

	for( int64_t f = first; f < fb; ++f, row_lo += M + 1, row_hi += M + 1, row_irr += M + 1 )
		{
		float2 v[PT];
			{
			const unsigned xb = ( (unsigned) t + (unsigned) T * (unsigned)( ( f + 8 ) & 15 ) ) * 8u;
#pragma unroll
			for( int s = 0; s < PT; ++s )
				{
				const float2 r = *reinterpret_cast<const float2 *>( reinterpret_cast<const char *>( ring ) + ( ( xb + (unsigned)( s * T * 8 ) ) & (unsigned)( 16 * T * 8 - 1 ) ) );
				float2 ww; ww.x = w[2 * s]; ww.y = w[2 * s + 1];
				v[s] = mul2( r, ww );
				}
			// entry of slot 0 is free now: it is slot 15 of the next frame
			*reinterpret_cast<float2 *>( reinterpret_cast<char *>( ring ) + xb ) = nxt;
			nxt = load_pair( f + 2, PT - 1 );
			}
		fft_butterflies<M, PT, PT, 1>( t, v, (const float2 *) nullptr, ldtw );
		fft_store<M, PT, PT, 1>( t, v, x0 );
		float2 tw[PT - 1];          // the next pass's twiddles, requested before the barrier (v is dead here)
		fft_load_twiddles<M, PT, PT, PT>( t, tw, a.pass_tw + P::tw_offset( 1 ), ldtw );
		env.sync();

		fft_load<M, PT, 1>( t, v, x0 );
		if( x0 == x1 ) env.sync();      // one exchange buffer: everyone has read before anyone writes
		fft_butterflies_w<M, PT, PT, PT>( v, tw );
		fft_store<M, PT, PT, PT>( t, v, x1 );
#pragma unroll
		for( int q = 0; q < Q; ++q )
#pragma unroll
			for( int r = 1; r < R; ++r ) tw[q * ( R - 1 ) + r - 1] = ldtw( tw_last + ( r - 1 ) * NS + t + q * T );
		env.sync();

		const bool emit = ( f >= fa );
#pragma unroll
		for( int q = 0; q < Q; ++q )
			{
			const int p = t + q * T;
			const bool irr = ( q == 0 ) && irregular;
			const int jA = p, jB = irr ? NS / 2 : NS - p;
			float2 * za = v + 2 * R * q, * zb = za + R;
#pragma unroll
			for( int r = 0; r < R; ++r ) { za[r] = x1[jA + r * NS]; zb[r] = x1[jB + r * NS]; }
			if( q == Q - 1 && x0 == x1 ) env.sync();    // one exchange buffer: the next frame's first pass writes it again
			// Twiddles of butterfly jB = NS - p': w^(r (NS - p')) = W_R^r conj(w^(r p')), p' = NS - jB (= p, or NS/2 for the
			// irregular thread). The factor W_R^r rotates the DFT by one bin (DFT_R{ u_r W_R^r }[k] = U[k+1]), so the
			// butterfly multiplies by the CONJUGATE of butterfly jA's twiddles -- no second table read except in the
			// warp of the irregular thread -- and its outputs are taken one register further on.
			const bool own_tw = ( q == 0 ) && warp0;                // warp-uniform
#pragma unroll
			for( int r = 1; r < R; ++r )
				{
				const float2 wa = tw[q * ( R - 1 ) + r - 1];
				float2 wb = wa;
				if( own_tw ) wb = ldtw( tw_last + ( r - 1 ) * NS + ( NS - jB ) );
				za[r] = cmul2( za[r], wa );
				zb[r] = cmulc2( zb[r], wb );
				}
			dft_r<R, 1>( za );
			dft_r<R, 1>( zb );
			// za[r] = Z[jA + r NS], zb[(r + 1) % R] = Z[jB + r NS]; slot r pairs Z[k], k = p + r NS, with Z[M-k] = Z[jB + (R-1-r) NS]
#pragma unroll
			for( int r = 0; r < R; ++r )
				{
				const int k = p + r * NS;
				const float2 zk = za[r], zm = zb[( R - r ) % R];
				const float2 A = add2( zk, pn2( zm ) );
				const float2 D = add2( zk, np2( zm ) );
				const float2 Pq = cmul2( D, env.ldg2( a.post_rot + k ) );
				const float2 xk = add2( A, Pq ), xmc = sub2( A, Pq );
				const float4 cc = env.ldg4( a.binc4 + k );
				float2 binf, expd; binf.x = cc.x; binf.y = cc.y; expd.x = cc.z; expd.y = cc.w;
				float2 mk, mm;
				phase_vocoder_pair( xk, xmc, prev[q][r], binf, expd, a.k, mk, mm );
				// the irregular thread's pairing is meaningless (its two butterflies are each their own mirror): see below
				if( emit && !irr )
					{
					env.st_stream2( row_lo + ( q * T + r * NS ), mk );
					env.st_stream2( row_hi - ( q * T + r * NS ), mm );
					}
				}
			// Bins that are multiples of NS/2 (2R+1 of them, 0 .. M): the irregular thread publishes its two butterflies,
			// scratch[j] = Z[(NS/2) j], and lanes 0..2R of its warp each finish one bin with the scalar form of the same
			// arithmetic: X[k] = (Z[k] + conj Z[M-k]) + (-i w_k)(Z[k] - conj Z[M-k]).
			if( q == 0 && warp0 )
				{
				if( irregular )
					{
#pragma unroll
					for( int r = 0; r < R; ++r ) { scratch[2 * r] = za[r]; scratch[2 * r + 1] = zb[( r + 1 ) % R]; }
					}
				env.syncwarp();
				if( t <= 2 * R )
					{
					const int k = ( NS / 2 ) * t;
					const float2 zk = scratch[t & ( 2 * R - 1 )], zm = scratch[( 2 * R - t ) & ( 2 * R - 1 )];
					const float2 A = add2( zk, pn2( zm ) );
					const float2 D = add2( zk, np2( zm ) );
					const float2 Pq = cmul2( D, env.ldg2( a.post_rot + k ) );
					const float2 xk = add2( A, Pq );
					const float2 ch = env.ldg2( a.binc + k );
					const float2 mh = phase_vocoder_bin( xk.x, xk.y, prev_irr, ch.x, ch.y, a.k );
					if( emit ) env.st_stream2( row_irr, mh );
					}
				}
			}
		}
	}

// ------------------------------------------------------------------------------------------------
// Resynthesis: phase-scan helpers
// ------------------------------------------------------------------------------------------------

// Segment summary of one bin over frames [fa,fb): total phase increment and its max prefix. Within a segment (a few
// thousand radians at most) the running sum is a plain double -- absolute error ~1e-12 rad -- and only the two
// results are converted to the split form (see PhaseSum). `flag` is raised on NaN/Inf, the is_nan_or_inf() pre-scan
// of AudioPV.cpp:88.
template<class Ld>
PV_HD PhaseSeg phase_segment_summary( const float2 * col, int64_t row_stride, int64_t rows, const PvConsts & k,
                                      double P, double rcpP, int & flag, Ld && ld )
	{
	PhaseSegAcc acc;
	int64_t i = 0;
	for( ; i + 8 <= rows; i += 8 )          // eight independent row loads in flight per thread
		{
		float2 mf[8];
#pragma unroll
		for( int j = 0; j < 8; ++j ) mf[j] = ld( col + ( i + j ) * row_stride );
#pragma unroll
		for( int j = 0; j < 8; ++j ) acc.step( mf[j], k );
		}
	for( ; i < rows; ++i ) acc.step( ld( col + i * row_stride ), k );
	if( acc.bad ) flag = 1;
	return acc.finish( P, rcpP );
	}

// state <- state (+) seg : running (sum, max prefix) over segments in frame order.
PV_HD void phase_state_combine( PhaseSeg & st, const PhaseSeg & seg, double P, double rcpP )
	{
	PhaseSum cand; cand.q = st.sum.q + seg.mx.q; cand.r = st.sum.r + seg.mx.r;
	phase_sum_normalize( cand, P, rcpP );
	if( phase_sum_less( st.mx, cand ) ) st.mx = cand;
	st.sum.q += seg.sum.q; st.sum.r += seg.sum.r;
	phase_sum_normalize( st.sum, P, rcpP );
	}

// The reference's accumulator value for running state st: S - P * max(0, floor(maxprefix / P)).
PV_HD double phase_state_value( const PhaseSeg & st, double P )
	{
	return fma( st.sum.q - st.mx.q, P, st.sum.r );
	}

// ------------------------------------------------------------------------------------------------
// Resynthesis
// ------------------------------------------------------------------------------------------------
struct SynthArgs
	{
	const float2 * pv;          // rows: pv + c * pv_channel_stride + (frame - frame_begin) * B
	int64_t pv_channel_stride;
	int64_t frame_begin, frame_end;
	float * out;                // local span; sample s of channel c at out + c * out_stride + (s - out_offset)
	int64_t out_stride;
	int64_t out_offset;
	int64_t out_lo, out_hi;     // absolute samples that exist in the local span (others are dropped: AudioPV.cpp:127-128)
	const double * acc_start;   // [C][segs_per_channel][B] accumulator value entering each segment
	int seg_len;
	int segs_per_channel;
	int seg_first, seg_count;   // this launch covers segments [seg_first, seg_first + seg_count) of every channel (0: all of them):
	                            // the pipelined host forms launch a signal in a few slices so that downloads can follow them
	int W, hop;
	int aligned2;
	const float * win;          // [W] Hann * window_scale, host-evaluated (AudioPV.cpp:99-102)
	const float2 * post_tw;
	const float2 * pass_tw;
	const float2 * pass_tw_rev; // twiddles of the small-radix-first plan (synthesis_cta_mirror)
	int out_aligned2;           // every even absolute sample of every channel sits on an 8-byte boundary of `out`
	int pv_aligned16;           // `pv` is 16-byte aligned (bulk row copies)
	int one_buffer;             // mirrored kernel: the two exchange buffers alias
	int channels;
	PvConsts k;
	double P, rcpP;             // double(pi2) and its reciprocal
	};

// ONE: the two exchange buffers alias (x1 == x0): three more barriers per frame, 37 KB less shared memory at dft 8192,
// which lets two CTAs share an SM there.
template<int N, bool ONE, class Env>
PV_HD void synthesis_cta( const SynthArgs & a, int64_t block, Env & env, float * ola, float2 * x0, float2 * x1, float2 * rowbuf )
	{
	constexpr int M = N / 2, T = M / 8, B = M + 1;
	const int t = env.tid;
	const int per_launch = a.seg_count > 0 ? a.seg_count : a.segs_per_channel;
	const int c = (int)( block / per_launch );
	const int seg = a.seg_first + (int)( block % per_launch );
	const int64_t fa = a.frame_begin + (int64_t) seg * a.seg_len;
	const int64_t fb = ( fa + a.seg_len < a.frame_end ) ? fa + a.seg_len : a.frame_end;
	if( fa >= fb ) return;

	const int W = a.W, hop = a.hop;
	const int half = W / 2;
	const int fin = ( hop < W ) ? hop : W;          // samples finalised per frame

	float w[16];
#pragma unroll
	for( int s = 0; s < 8; ++s )
		{
		const int i0 = 2 * ( t + s * T );
		w[2 * s]     = ( i0 < W )     ? env.ldg( a.win + i0 ) : 0.0f;
		w[2 * s + 1] = ( i0 + 1 < W ) ? env.ldg( a.win + i0 + 1 ) : 0.0f;
		}
	double acc[9];
	const double * acc0 = a.acc_start + ( (int64_t) c * a.segs_per_channel + seg ) * B;
#pragma unroll
	for( int u = 0; u < 4; ++u )
		{
		const int k = t + u * T;
		acc[2 * u] = acc0[k];
		acc[2 * u + 1] = acc0[M - k];
		}
	acc[8] = acc0[M / 2];

	for( int i = t; i < N; i += T ) ola[i] = 0.0f;

	// The (m,f) row of the NEXT frame is staged into shared memory with 8-byte cp.async while the current frame
	// computes, so the HBM latency of the streaming read never sits on the critical path.
	const float2 * pv_ch = a.pv + (int64_t) c * a.pv_channel_stride;
	auto stage_row = [&]( int64_t f )
		{
		const float2 * src = pv_ch + ( f - a.frame_begin ) * (int64_t) B;
		for( int i = t; i < B; i += T ) env.cp_async8( rowbuf + i, src + i );
		env.cp_async_commit();
		};
	stage_row( fa );
	env.cp_async_wait_all();
	env.sync();

	float * och = a.out + (int64_t) c * a.out_stride;
	// Samples whose every contributing frame lies in this segment are stored; the W-hop samples shared with
	// the previous / next segment receive exactly two partial sums and are combined with red.add (a + b is
	// commutative, so the result does not depend on arrival order).
	const int64_t interior_lo = (int64_t) hop * fa + half - hop;
	const int64_t interior_hi = (int64_t) hop * fb - half;
	auto flush = [&]( int64_t lo, int64_t hi )
		{
		if( lo >= interior_lo && hi <= interior_hi && lo >= a.out_lo && hi <= a.out_hi )
			{
			// whole range final and inside the local span (every frame but the first and last W/hop of a segment)
			float * dst = och + ( lo - a.out_offset );
			const int rs0 = (int) lo & ( N - 1 );
			for( int i = t; i < (int)( hi - lo ); i += T )
				{
				const int slot = ( rs0 + i ) & ( N - 1 );
				env.st_stream( dst + i, ola[slot] );
				ola[slot] = 0.0f;
				}
			return;
			}
		for( int64_t s = lo + t; s < hi; s += T )
			{
			const int slot = (int) s & ( N - 1 );
			const float val = ola[slot];
			ola[slot] = 0.0f;
			if( s >= a.out_lo && s < a.out_hi )
				{
				float * dst = och + ( s - a.out_offset );
				if( s >= interior_lo && s < interior_hi ) env.st_stream( dst, val );
				else env.red_add( dst, val );
				}
			}
		};

	auto polar = [&]( float2 mf, double & ph ) -> float2
		{
#ifndef PV_ABL_NOEPI
		phase_accumulate( ph, phase_increment( mf.y, a.k ), a.P, a.rcpP );      // phase_vocoder.cpp:57-59
		const float theta = (float) ph;
		float sn, cs;
		sincos_pv( theta, &sn, &cs );
		float2 r; r.x = mul_rn( mf.x, cs ); r.y = mul_rn( mf.x, sn );           // :60 std::polar
		return r;
#else
		return mf;                                                              // ablation build only
#endif
		};

	const bool full_window = ( W == N ) && a.aligned2;
	for( int64_t f = fa; f < fb; ++f )
		{
		const int64_t start = (int64_t) hop * f - half;                          // AudioPV.cpp:125
		const float2 * row = rowbuf;

		// bins -> packed half-size spectrum Z'[k] = (X[k] + conj X[M-k]) + i e^{+2 pi i k/N} (X[k] - conj X[M-k]),
		// stored with re/im swapped so the forward pass chain computes the inverse transform.
		float2 v[8];
#pragma unroll
		for( int u = 0; u < 4; ++u )
			{
			const int k = t + u * T;
			float2 xk, xm;
#ifndef PV_ABL_NOEPI
			inverse_pv_pair( row[k], row[M - k], acc[2 * u], acc[2 * u + 1], a.k, a.P, a.rcpP, xk, xm );
#else
			xk = row[k]; xm = row[M - k];                                   // ablation build only
#endif
			// imaginary parts of bins 0 and N/2 are ignored by a c2r transform: with them cleared the general pack gives
			// Z'[0] = (X0 + XM) + i (X0 - XM); its mirror lands in the unused slot M of the buffer
			if( u == 0 && t == 0 ) { xk.y = 0.0f; xm.y = 0.0f; }
			// A = X[k] + conj X[M-k], Bv = X[k] - conj X[M-k], Q = Bv * conj(w_k); Z'[k] = A + iQ, Z'[M-k] = conj(A - iQ),
			// both stored with (im, re) swapped.
			const float2 tw = env.ldg2( a.post_tw + k );
			const float2 A = add2( xk, pn2( xm ) );
			const float2 Bv = add2( xk, np2( xm ) );
			const float2 Q = cmulc2( Bv, tw );
			v[u] = add2( swap2( A ), pn2( Q ) );            // Z'[t + u*T] is this thread's own pass-0 input
			x1[M - k] = add2( np2( swap2( A ) ), Q );       // the mirror side belongs to thread T - t
			}
		if( t == T / 2 )
			{
			const float2 xh = polar( row[M / 2], acc[8] );
			float2 zs; zs.y = 2.0f * xh.x; zs.x = -2.0f * xh.y;   // Z'[M/2] = 2 conj X[M/2], swapped
			x1[M / 2] = zs;
			}
		env.sync();

		// every thread has consumed its bins of this row: start fetching the next one
		if( f + 1 < fb ) stage_row( f + 1 );

#pragma unroll
		for( int s = 4; s < 8; ++s ) v[s] = x1[t + s * T];          // upper half of Z' from the mirror threads
		if constexpr( ONE ) env.sync();
		fft_butterflies<M, 8, 8, 1>( t, v, (const float2 *) nullptr, [&]( const float2 * q ) { return env.ldg2( q ); } );
		fft_store<M, 8, 8, 1>( t, v, x0 );
		float2 tw[7];
		fft_chain_twiddles<M, 8, 1>( t, tw, a.pass_tw, env );
		env.sync();
#ifndef PV_ABL_NOFFT
		fft_pass_chain<M, 8, 1, false, ONE, true>( t, v, x0, x1, a.pass_tw, env, tw );
#endif

		// v[s] = swapped z[n], n = t + s*T: y[2n] = v.y, y[2n+1] = v.x. Windowed overlap-add (AudioPV.cpp:133-134).
		const int rs = (int) start & ( N - 1 );
#ifdef PV_ABL_NOOLA
		if( v[0].x == 123.456f )                                              // ablation build only
#endif
		if( full_window )
			{
			// whole window, even ring positions: out += y * w as one packed multiply and one packed add per sample pair
			// (each lane rounds like the scalar mul_rn / add_rn: no contraction)
#pragma unroll
			for( int s = 0; s < 8; ++s )
				{
				float2 * slot = reinterpret_cast<float2 *>( ola + ( ( rs + 2 * ( t + s * T ) ) & ( N - 1 ) ) );
				float2 ww; ww.x = w[2 * s]; ww.y = w[2 * s + 1];
				*slot = add2( *slot, mul2( swap2( v[s] ), ww ) );
				}
			}
		else if( a.aligned2 )
			{
#pragma unroll
			for( int s = 0; s < 8; ++s )
				{
				const int i0 = 2 * ( t + s * T );
				if( i0 < W )
					{
					float2 * slot = reinterpret_cast<float2 *>( ola + ( ( rs + i0 ) & ( N - 1 ) ) );
					float2 cur = *slot;
					cur.x = add_rn( cur.x, mul_rn( v[s].y, w[2 * s] ) );
					if( i0 + 1 < W ) cur.y = add_rn( cur.y, mul_rn( v[s].x, w[2 * s + 1] ) );
					*slot = cur;
					}
				}
			}
		else
			{
#pragma unroll
			for( int s = 0; s < 8; ++s )
				{
				const int i0 = 2 * ( t + s * T );
				if( i0 < W )
					{
					float * p0 = ola + ( ( rs + i0 ) & ( N - 1 ) );
					*p0 = add_rn( *p0, mul_rn( v[s].y, w[2 * s] ) );
					}
				if( i0 + 1 < W )
					{
					float * p1 = ola + ( ( rs + i0 + 1 ) & ( N - 1 ) );
					*p1 = add_rn( *p1, mul_rn( v[s].x, w[2 * s + 1] ) );
					}
				}
			}
		env.cp_async_wait_all();       // the next row has had the whole pass chain to arrive; the barrier publishes it
		env.sync();
		// no later frame of this segment reaches [start, start+fin) again; the barriers of the next
		// frame order this zeroing before its overlap-add
		flush( start, start + fin );
		}
	// remainder of the last window
	const int64_t last_start = (int64_t) hop * ( fb - 1 ) - half;
	flush( last_start + fin, last_start + W );
	}

// ------------------------------------------------------------------------------------------------
// Resynthesis, mirrored first pass (16 points per thread; dft 1024 / 2048 / 4096, window == dft, hop a multiple of
// dft/16). The transpose of analysis_cta_mirror: the inverse FFT runs as passes R, 16, 16 (R = 2 / 4 / 8), and one
// thread computes the two first-pass butterflies p and NS-p, whose inputs Z'[p + r NS] and Z'[(NS-p) + r NS] are
// exactly the packed values of the bin pairs (k, M-k), k = p + r NS. So a thread reads ITS OWN bins of the row,
// accumulates their phases in registers, packs and transforms them without any exchange, and
//   * the (m,f) row is a thread-private prefetch FIFO in shared memory: every thread stages (8-byte cp.async) and
//     reads only its own 2R+1 bins, so no barrier guards it;
//   * with hop == j * dft/16 the overlap-add positions of a thread are the same absolute samples in every frame
//     (pair index mod T == t), so the ring is thread-private as well: no barrier, and the `hop` samples a frame
//     finalises are the thread's slots s < j, which go from registers straight to global memory.
// Two barriers per frame remain: the two FFT exchanges. Contributions are added in increasing frame order
// (AudioPV.cpp:133-134), every product and sum rounded separately, exactly like synthesis_cta.
// ------------------------------------------------------------------------------------------------
template<int M, int R> struct RevPlan
	{
	// Stockham passes R, 16, 16 (and a last radix-2 pass at 4096 points) of a complex M-point FFT, 16 points per thread
	static constexpr int NS1 = R, NS2 = 16 * R, NS3 = 256 * R;
	static constexpr int R3 = M / NS3;             // 1 (no fourth pass) or 2
	static_assert( R3 == 1 || R3 == 2, "M = 256 R or 512 R" );
	static constexpr int tw1 = 0;                  // pass 1 (radix 16, Ns = R):    [15][R]
	static constexpr int tw2 = 15 * NS1;           // pass 2 (radix 16, Ns = 16R):  [15][16R]
	static constexpr int tw3 = tw2 + 15 * NS2;     // pass 3 (radix 2, Ns = 256R):  [1][256R]
	static constexpr int tw_total = tw3 + ( R3 - 1 ) * NS3;
	};

// Exchange layout after the radix-16 pass with Ns = R (lanes write 16R*(jj/R) + jj%R + R*r): blocks of 16R elements
// are shifted by R each, which makes the 16 accesses of a half-warp hit 16 distinct 8-byte bank pairs; the reads
// t + s*T of the next pass (T a multiple of 16R) stay contiguous per half-warp.
template<int R> PV_HD int xpad_rev( int i ) { return i + R * ( i / ( 16 * R ) ); }

// Exchange layout after the mirrored first pass of radix 8: a thread stores the 8 outputs of butterfly p at 8p + r
// (ascending with the lane) and those of butterfly NS - p at 8(NS - p) + r (descending). With the plain xpad<1> the
// descending stores of a half-warp span 128 padded elements exactly -- its first and last lane meet in one bank pair and
// every such store takes twice the wavefronts (ncu, round 1: all 33.9 M excess wavefronts of the kernel, 14.5 % of its
// shared-memory traffic, sat on these eight STS.64). The pad g(u) of each aligned group u of 16 elements must satisfy,
// for lanes of even p (bank-pair index g(u) mod 16) and odd p (8 + g(u) mod 16) alike, g(u) mod 16 in [0, 8) and
// distinct for eight consecutive u in ANY alignment: g(u) = (u & 7) + 16 (u >> 3), 247 pad elements of the M/8 = 256
// the buffer has at dft 4096. Groups of 16 stay contiguous, so the next pass's reads t + s*T keep their layout
// (pad( t + s*T ) = pad( t ) + pad( s*T ) for T = 128 and 256).
template<int R> PV_HD int mpad( int i )
	{
	if( R == 8 ) return i + ( ( i >> 4 ) & 7 ) + ( ( i >> 7 ) << 4 );
	return xpad<1>( i );
	}

// ONE: the two exchange buffers alias (x1 == x0): two more barriers per frame, 18 KB less shared memory per CTA, which
// moves the SM's carve-out from 228 KB to 164 KB and so gives the twiddle tables (32 KB) an L1 they fit in.
// GEN: any window that fills whole slots of the thread layout (a multiple of dft/16 samples) and any even hop up to
// dft/16 -- e.g. the API default window 2048 / hop 128 / dft 4096 (Audio.h:158-163). A frame then advances the
// overlap-add positions by hop/2 pairs, which is no longer a whole slot per thread, so the ring is shared by the CTA (the
// two exchange barriers of the next frame order one frame's accumulation before the next one's; no barrier is added),
// and whether a thread's last used slot starts a ring entry and whether its slot 0 is final depends on the thread (two
// predicates, fixed over the walk). !GEN is the standard shape (window == dft, hop == dft/16) with everything resolved at compile time.
// Tensor memory of the mirrored resynthesis at dft 4096, standard shape (128 threads, thread t owns lane t, 128 columns per
// CTA: four CTAs per SM at 128 registers use all 512):
//   columns  0..31  window coefficients w[0..31]
//           32..47  post_tw[k] of the thread's 8 bins (slot r at 32 + 2r)
//           48..77  the 15 twiddles of the second radix-16 pass (78..95 zero)
//           96..125 the overlap-add partials: R[j] at 96 + 2j, j = 0..14, the partial sum of slot j of the next frame
//                   (126..127 zero)
// The window is read once per frame, for the overlap-add; the first pass's twiddles stay in L1 (index t mod 8). The
// partials replace the shared-memory ring of the other sizes: slot s of frame f is slot s-1 of frame f+1, so instead of
// a rotating address the sums move down one column pair per frame, a renaming fixed at compile time.
template<int N, bool GEN> constexpr bool synthesis_tmem() { return N == 4096 && !GEN; }
constexpr int SY_TM_COLS = 128, SY_TM_WIN = 0, SY_TM_POST = 32, SY_TM_TW = 48, SY_TM_OLA = 96;

// TM: the tensor-memory form (synthesis_tmem); the Env then addresses the CTA's SY_TM_COLS columns.
template<int N, bool ONE, bool GEN, bool TM = synthesis_tmem<N, GEN>(), class Env>
PV_HD void synthesis_cta_mirror( const SynthArgs & a, int64_t block, Env & env, float2 * ring, float2 * x0, float2 * x1, float2 * rowbuf,
                                 typename Env::BulkBarrier * bar )
	{
	using MP = MirrorPlan<N>;
	constexpr int PT = 16, M = MP::M, T = MP::T, R = MP::R, NS = MP::NS, Q = MP::Q, B = M + 1;
	using RP = RevPlan<M, R>;
	static_assert( T % ( 16 * R ) == 0, "threads per frame" );
	static_assert( !TM || ( T == 128 && Q == 1 && R == 8 && RP::R3 == 1 && !GEN ), "tensor-memory layout of the dft-4096 resynthesis" );
	const int t = env.tid;
	const int per_launch = a.seg_count > 0 ? a.seg_count : a.segs_per_channel;
	const int c = (int)( block / per_launch );
	const int seg = a.seg_first + (int)( block % per_launch );
	const int64_t fa = a.frame_begin + (int64_t) seg * a.seg_len;
	const int64_t fb = ( fa + a.seg_len < a.frame_end ) ? fa + a.seg_len : a.frame_end;
	if( fa >= fb ) return;

	const int hop = GEN ? a.hop : 2 * T;         // !GEN: == a.hop == N/16 and window == N
	const int half = GEN ? a.W / 2 : N / 2;
	const int wp = half;                         // window length in sample pairs
	const int hp = hop / 2;                      // pairs a frame advances by
	const bool irregular = ( t == 0 );
	const int khi = irregular ? MP::KHI : 0;

	float w[2 * PT];
	// GEN (hop <= dft/16, i.e. hp <= T): slot s of this thread is pair n = t + s*T of the frame's window. Slots
	// s < slots_in are used; of the last used slot the pairs n >= wp - hp are `fresh` (this is the first frame to reach
	// their absolute pair: the ring entry is overwritten), of slot 0 the pairs n < hp are `final` (no later frame reaches
	// them: they go straight to global memory). Both are ranges of t, uniform per warp when hp is a multiple of 32.
	const int slots_in = GEN ? wp / T : PT;
	const bool is_final = GEN ? ( t < hp ) : true;
	const bool is_fresh = GEN ? ( t >= T - hp ) : true;
#pragma unroll
	for( int s = 0; s < PT; ++s )
		{
		const int nn = t + s * T;
		if( !GEN || nn < wp )
			{
			w[2 * s]     = env.ldg( a.win + 2 * nn );
			w[2 * s + 1] = env.ldg( a.win + 2 * nn + 1 );
			}
		else { w[2 * s] = 0.0f; w[2 * s + 1] = 0.0f; }
		}
	// TM: the tables go to tensor memory before the accumulators are loaded; with all three live at once ptxas keeps four
	// accumulators in local memory for the whole frame loop
	if constexpr( TM )
		{
		env.template tmem_st<32>( SY_TM_WIN, w );
		float2 tb[32];              // columns 32..95: post_tw, the pass twiddles, zeros
#pragma unroll
		for( int r = 0; r < R; ++r ) tb[r] = env.ldg2( a.post_tw + ( t + ( ( r >= R / 2 ) ? khi : 0 ) + r * NS ) );
		fft_load_twiddles<M, PT, PT, RP::NS2>( t, tb + 8, a.pass_tw_rev + RP::tw2, [&]( const float2 * q ) { return env.ldg2( q ); } );
#pragma unroll
		for( int i = 23; i < 32; ++i ) { tb[i].x = 0.0f; tb[i].y = 0.0f; }
		env.template tmem_st<32>( SY_TM_POST, reinterpret_cast<const float *>( tb ) );
		env.template tmem_st<32>( SY_TM_POST + 32, reinterpret_cast<const float *>( tb + 16 ) );
#pragma unroll
		for( int i = 0; i < 16; ++i ) { tb[i].x = 0.0f; tb[i].y = 0.0f; }
		env.template tmem_st<32>( SY_TM_OLA, reinterpret_cast<const float *>( tb ) );
		env.tmem_wait_st();
		}
	else
		{
		// thread-private overlap-add ring: 16 pairs at ring[t + T*j]; absolute pair index t + T*A lives in slot A & 15
#pragma unroll
		for( int j = 0; j < PT; ++j ) { float2 z; z.x = 0.0f; z.y = 0.0f; ring[t + T * j] = z; }
		}

	// bin of slot (q, r): k = kbase + r*NS with kbase = p (+ khi for the irregular upper slots); its mirror is M - k
	double acc[Q][R][2], acc_mid = 0.0;
	const double * acc0 = a.acc_start + ( (int64_t) c * a.segs_per_channel + seg ) * B;
#pragma unroll
	for( int q = 0; q < Q; ++q )
#pragma unroll
		for( int r = 0; r < R; ++r )
			{
			const int k = t + q * T + ( ( q == 0 && r >= R / 2 ) ? khi : 0 ) + r * NS;
			acc[q][r][0] = acc0[k];
			acc[q][r][1] = acc0[M - k];
			}
	if( irregular ) acc_mid = acc0[M / 2];
	// Row staging. A row is 8 B * (M+1) long and only 8-byte aligned, so the bulk (TMA) copy fetches the enclosing
	// 16-byte aligned span -- at most one (m,f) pair of a neighbouring row on either side -- and the row starts `shift`
	// elements into the buffer. One thread issues it, completion arrives on an mbarrier. Where the span would leave
	// the PV buffer (its very last row) or the buffer is not 16-byte aligned, every thread copies its own bins with
	// 8-byte cp.async instead.
	const float2 * pv_ch = a.pv + (int64_t) c * a.pv_channel_stride;
	const int64_t pv_end = (int64_t)( a.channels - 1 ) * a.pv_channel_stride + ( a.frame_end - a.frame_begin ) * (int64_t) B;   // elements in the buffer
	auto row_elem = [&]( int64_t f ) { return (int64_t) c * a.pv_channel_stride + ( f - a.frame_begin ) * (int64_t) B; };
	auto row_is_bulk = [&]( int64_t f )
		{
		const int64_t e = row_elem( f );
		return a.pv_aligned16 && ( ( ( e + B + 1 ) & ~(int64_t) 1 ) <= pv_end );
		};
	auto stage_row_own = [&]( int64_t f )
		{
		const float2 * src = pv_ch + ( f - a.frame_begin ) * (int64_t) B;
#pragma unroll 1
		for( int i = 0; i < 2 * R * Q; ++i )
			{
			const int q = i / ( 2 * R ), r = ( i / 2 ) % R;
			int k = t + q * T + ( ( q == 0 && r >= R / 2 ) ? khi : 0 ) + r * NS;
			if( i & 1 ) k = M - k;
			env.cp_async8( rowbuf + k, src + k );
			}
		if( irregular ) env.cp_async8( rowbuf + M / 2, src + M / 2 );
		env.cp_async_commit();
		};
	auto stage_row_bulk = [&]( int64_t f )       // one thread
		{
		const int64_t e = row_elem( f ), e0 = e & ~(int64_t) 1, e1 = ( e + B + 1 ) & ~(int64_t) 1;
		env.bulk_load( rowbuf, a.pv + e0, (unsigned)( ( e1 - e0 ) * sizeof( float2 ) ), bar );
		};
	if( t == 0 ) env.bulk_init( bar );
	env.sync();
	unsigned bulk_phase = 0;
	bool cur_bulk = row_is_bulk( fa );
	if( cur_bulk ) { if( t == 0 ) stage_row_bulk( fa ); }
	else stage_row_own( fa );

	float * och = a.out + (int64_t) c * a.out_stride;
	const int64_t interior_lo = (int64_t) hop * fa + half - hop;
	const int64_t interior_hi = (int64_t) hop * fb - half;
	// one finished sample: stored when every contributing frame lies in this segment, else combined with the
	// neighbouring segment's partial sum by red.add (exactly two partial sums meet; a + b is commutative)
	auto emit = [&]( int64_t pos, float val )
		{
		if( pos >= a.out_lo && pos < a.out_hi )
			{
			float * dst = och + ( pos - a.out_offset );
			if( pos >= interior_lo && pos < interior_hi ) env.st_stream( dst, val );
			else env.red_add( dst, val );
			}
		};
	auto ldtw = [&]( const float2 * q ) { return env.ldg2( q ); };

	for( int64_t f = fa; f < fb; ++f )
		{
		const int64_t start = (int64_t) hop * f - half;                          // AudioPV.cpp:125
		const float2 * row = rowbuf;
		float2 ptw[R];              // TM: post_tw of the thread's bins
		if constexpr( TM ) env.template tmem_ld<2 * R>( SY_TM_POST, reinterpret_cast<float *>( ptw ) );
		if( cur_bulk ) { env.bulk_wait( bar, bulk_phase & 1 ); ++bulk_phase; row = rowbuf + ( row_elem( f ) & 1 ); }
		else env.cp_async_wait_all();                                            // this thread's bins of row f have landed
		if constexpr( TM ) env.template tmem_wait<2 * R>( reinterpret_cast<float *>( ptw ) );
		float2 v[PT];
#pragma unroll
		for( int q = 0; q < Q; ++q )
			{
			const int p = t + q * T;
			const bool irr = ( q == 0 ) && irregular;
			float2 zk[R], zm[R];
#pragma unroll
			for( int r = 0; r < R; ++r )
				{
				const int k = p + ( ( q == 0 && r >= R / 2 ) ? khi : 0 ) + r * NS;
				float2 xk, xm;
				inverse_pv_pair( row[k], row[M - k], acc[q][r][0], acc[q][r][1], a.k, a.P, a.rcpP, xk, xm );
				// a c2r transform ignores the imaginary parts of bins 0 and N/2 (slot 0 of the irregular pair)
				if( r == 0 && irr ) { xk.y = 0.0f; xm.y = 0.0f; }
				const float2 tw = TM ? ptw[r] : env.ldg2( a.post_tw + k );
				const float2 A = add2( xk, pn2( xm ) );
				const float2 Bv = add2( xk, np2( xm ) );
				const float2 Qv = cmulc2( Bv, tw );
				zk[r] = add2( swap2( A ), pn2( Qv ) );            // Z'[k], (im, re) swapped: the forward passes then invert
				zm[r] = add2( np2( swap2( A ) ), Qv );            // Z'[M-k]
				}
			float2 * za = v + 2 * R * q, * zb = za + R;
#pragma unroll
			for( int r = 0; r < R; ++r ) { za[r] = zk[r]; zb[R - 1 - r] = zm[r]; }
			if( irr )
				{
				// butterflies 0 and NS/2 take their inputs in another arrangement, plus bin M/2
				float sn, cs;
				const float2 mh = row[M / 2];
				phase_accumulate( acc_mid, phase_increment( mh.y, a.k ), a.P, a.rcpP );      // phase_vocoder.cpp:57-59
				sincos_pv( (float) acc_mid, &sn, &cs );
				float2 zs; zs.y = 2.0f * mul_rn( mh.x, cs ); zs.x = -2.0f * mul_rn( mh.x, sn );   // Z'[M/2] = 2 conj X[M/2], swapped
#pragma unroll
				for( int r = 0; r < R; ++r )
					{
					if( r < R / 2 ) { za[r] = zk[r]; if( r > 0 ) za[R - r] = zm[r]; }
					else            { zb[r - R / 2] = zk[r]; zb[3 * R / 2 - 1 - r] = zm[r]; }
					}
				za[R / 2] = zs;
				}
			}
		// pass 0: radix R, no twiddles, butterflies p and NS-p; outputs R*jj + r in the padded layout
		// the previous frame's last pass has read this buffer (long ago: the barrier is cheap); with the fourth pass of
		// dft 8192 that holds for x0 even when the two buffers are distinct
		if constexpr( ONE || RP::R3 > 1 ) env.sync();
#pragma unroll
		for( int q = 0; q < Q; ++q )
			{
			const int p = t + q * T;
			const int jA = p, jB = ( q == 0 && irregular ) ? NS / 2 : NS - p;
			float2 * za = v + 2 * R * q, * zb = za + R;
			dft_r<R, 1>( za );
			dft_r<R, 1>( zb );
			float2 * oa = x0 + mpad<R>( R * jA ), * ob = x0 + mpad<R>( R * jB );
#pragma unroll
			for( int r = 0; r < R; ++r ) { oa[r] = za[r]; ob[r] = zb[r]; }
			}
		float2 tw[PT - 1];          // the next pass's twiddles, requested before the barrier (v is dead here)
		fft_load_twiddles<M, PT, PT, RP::NS1>( t, tw, a.pass_tw_rev + RP::tw1, ldtw );
		env.sync();
		// every thread has consumed row f: fetch row f+1 behind the transform
		const bool next_bulk = ( f + 1 < fb ) && row_is_bulk( f + 1 );
		if( f + 1 < fb )
			{
			if( next_bulk ) { if( t == 0 ) stage_row_bulk( f + 1 ); }
			else stage_row_own( f + 1 );
			}
		cur_bulk = next_bulk;
		// pass 1: radix 16, Ns = R
			{
			const float2 * base = x0 + mpad<R>( t );
#pragma unroll
			for( int s = 0; s < PT; ++s ) v[s] = base[mpad<R>( s * T )];
			}
		if constexpr( ONE ) env.sync();     // everyone has read before anyone writes
		fft_butterflies_w<M, PT, PT, RP::NS1>( v, tw );
			{
			const int base = xpad_rev<R>( ( t / R ) * R * PT + ( t & ( R - 1 ) ) );
#pragma unroll
			for( int r = 0; r < PT; ++r ) x1[base + r * R] = v[r];
			}
		if constexpr( TM )
			{
			float * twf = reinterpret_cast<float *>( tw );
			env.template tmem_ld<16>( SY_TM_TW, twf );
			env.template tmem_ld<8>( SY_TM_TW + 16, twf + 16 );
			env.template tmem_ld<4>( SY_TM_TW + 24, twf + 24 );
			env.template tmem_ld<2>( SY_TM_TW + 28, twf + 28 );
			}
		else fft_load_twiddles<M, PT, PT, RP::NS2>( t, tw, a.pass_tw_rev + RP::tw2, ldtw );
		env.sync();
		// pass 2: radix 16, Ns = 16R. Without a fourth pass (T == 16R) its outputs are t + r*T, i.e. v[s] = swapped z[t + s*T]:
		// y[2n] = v.y, y[2n+1] = v.x
			{
			const float2 * base = x1 + xpad_rev<R>( t );
#pragma unroll
			for( int s = 0; s < PT; ++s ) v[s] = base[s * ( T + R * ( T / ( 16 * R ) ) )];
			}
		if constexpr( ONE && RP::R3 > 1 ) env.sync();       // everyone has read before anyone writes
		if constexpr( TM )
			{
			env.template tmem_wait<2 * ( PT - 1 )>( reinterpret_cast<float *>( tw ) );
			env.template tmem_ld<2 * PT>( SY_TM_WIN, w );      // this frame's window, for the overlap-add
			}
		fft_butterflies_w<M, PT, PT, RP::NS2>( v, tw );
		if constexpr( RP::R3 > 1 )
			{
			// pass 3 (dft 8192): radix 2, Ns = 256R, eight butterflies per thread; outputs in natural order
			float2 * xo = ONE ? x1 : x0;
				{
				const int base = ( t / RP::NS2 ) * RP::NS2 * PT + ( t & ( RP::NS2 - 1 ) );
#pragma unroll
				for( int r = 0; r < PT; ++r ) xo[base + r * RP::NS2] = v[r];
				}
			fft_load_twiddles<M, PT, RP::R3, RP::NS3>( t, tw, a.pass_tw_rev + RP::tw3, ldtw );
			env.sync();
#pragma unroll
			for( int s = 0; s < PT; ++s ) v[s] = xo[t + s * T];
			fft_butterflies_w<M, PT, RP::R3, RP::NS3>( v, tw );
			}

		// windowed overlap-add (AudioPV.cpp:133-134)
		float2 sum[PT];
		if constexpr( TM )
			{
			// TM: sum[s] = R[s] + prod[s], sum[15] = prod[15], then R[s-1] = sum[s]. R is read in x8 chunks of four slots (the
			// last one ends in the zero columns 126..127), each requested one chunk ahead, and written back in x8 chunks as soon
			// as the four sums of one are complete: 30 more live registers at once would not fit. The stores of this frame are
			// waited for (wait::st) before the next frame reads the columns, long after they were issued.
			float rb[2][8];
			env.tmem_wait_st();
			env.template tmem_ld<8>( SY_TM_OLA, rb[0] );
			env.template tmem_wait<2 * PT>( w );
			env.template tmem_wait<8>( rb[0] );
#pragma unroll
			for( int c = 0; c < PT / 4; ++c )
				{
				if( c > 0 ) env.template tmem_wait<8>( rb[c & 1] );
				if( c + 1 < PT / 4 ) env.template tmem_ld<8>( SY_TM_OLA + 8 * ( c + 1 ), rb[( c + 1 ) & 1] );
#pragma unroll
				for( int j = 0; j < 4; ++j )
					{
					const int s = 4 * c + j;
					float2 ww; ww.x = w[2 * s]; ww.y = w[2 * s + 1];
					const float2 prod = mul2( swap2( v[s] ), ww );
					float2 cur; cur.x = rb[c & 1][2 * j]; cur.y = rb[c & 1][2 * j + 1];
					sum[s] = ( s == PT - 1 ) ? prod : add2( cur, prod );
					}
				if( c > 0 ) env.template tmem_st<8>( SY_TM_OLA + 8 * ( c - 1 ), reinterpret_cast<const float *>( sum + 4 * c - 3 ) );
				}
			env.template tmem_st<4>( SY_TM_OLA + 24, reinterpret_cast<const float *>( sum + 13 ) );
			env.template tmem_st<2>( SY_TM_OLA + 28, reinterpret_cast<const float *>( sum + 15 ) );
			}
		else
			{
			// !GEN: on the thread's own ring; slot s of this frame is absolute pair t + T*(f + s - 8) (half/2 == 8T), i.e. ring
			// entry (f + s + 8) & 15 (byte offsets: (t + T*((f + 8 + s) & 15)) * 8 == ((t + T*(f + 8)) * 8 + s*T*8) & (16*T*8 - 1),
			// one add and one mask per slot).
			// GEN: absolute pair hp*f - wp/2 + t + s*T, ring entry that modulo 16T (the ring holds dft/2 >= wp pairs).
			const unsigned xb = GEN ? (unsigned)( ( (int64_t) hp * f - wp / 2 + t + (int64_t) PT * T * 4096 ) & (int64_t)( PT * T - 1 ) ) * 8u
			                        : ( (unsigned) t + (unsigned) T * (unsigned)( ( f + 8 ) & 15 ) ) * 8u;
			auto slot = [&]( int s ) { return reinterpret_cast<float2 *>( reinterpret_cast<char *>( ring ) + ( ( xb + (unsigned)( s * T * 8 ) ) & (unsigned)( 16 * T * 8 - 1 ) ) ); };
#pragma unroll
			for( int s = 0; s < PT; ++s )
				{
				float2 ww; ww.x = w[2 * s]; ww.y = w[2 * s + 1];
				const float2 prod = mul2( swap2( v[s] ), ww );
				// a fresh slot receives its first contribution (its ring entry is simply overwritten)
				if( GEN )
					{
					float2 cur; cur.x = 0.0f; cur.y = 0.0f;
					if( s < slots_in ) cur = *slot( s );                       // uniform over the CTA
					sum[s] = ( s == slots_in - 1 && is_fresh ) ? prod : add2( cur, prod );
					}
				else sum[s] = ( s == PT - 1 ) ? prod : add2( *slot( s ), prod );
				}
#pragma unroll
			for( int s = 1; s < PT; ++s ) if( !GEN || s < slots_in ) *slot( s ) = sum[s];
			if( !is_final ) *slot( 0 ) = sum[0];
			}
		if( is_final )
			{
			// slot 0: no later frame reaches these two samples
			const bool fast = start >= interior_lo && start + hop <= interior_hi && start >= a.out_lo && start + hop <= a.out_hi && a.out_aligned2;
			const int64_t pos = start + 2 * t;
			if( fast ) env.st_stream2( reinterpret_cast<float2 *>( och + ( pos - a.out_offset ) ), sum[0] );
			else { emit( pos, sum[0].x ); emit( pos + 1, sum[0].y ); }
			}
		}
	// remainder of the last window
	const int64_t last_start = (int64_t) hop * ( fb - 1 ) - half;
	if( GEN )
		{
		env.sync();                 // the ring entries read here were written by other threads in the last frame
		const unsigned xl = (unsigned)( ( (int64_t) hp * ( fb - 1 ) - wp / 2 + t + (int64_t) PT * T * 4096 ) & (int64_t)( PT * T - 1 ) );
#pragma unroll 1
		for( int s = 0; s < PT; ++s )
			{
			const int nn = t + s * T;
			if( nn < hp || nn >= wp ) continue;
			const float2 val = ring[( xl + (unsigned)( s * T ) ) & (unsigned)( PT * T - 1 )];
			const int64_t pos = last_start + 2 * nn;
			emit( pos, val.x ); emit( pos + 1, val.y );
			}
		return;
		}
	const int j0 = (int)( ( ( fb - 1 ) + 8 ) & 15 );
	if constexpr( TM ) env.tmem_wait_st();
#pragma unroll 1
	for( int s = 1; s < PT; ++s )
		{
		float2 val;
		if constexpr( TM )
			{
			float r[2];
			env.template tmem_ld<2>( SY_TM_OLA + 2 * ( s - 1 ), r );
			env.template tmem_wait<2>( r );
			val.x = r[0]; val.y = r[1];
			}
		else val = ring[t + T * ( ( j0 + s ) & 15 )];
		const int64_t pos = last_start + 2 * ( t + s * T );
		emit( pos, val.x ); emit( pos + 1, val.y );
		}
	}

} // namespace pvk
