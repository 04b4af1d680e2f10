// flan_b200/csrc/pv_policy.h -- the launch policy of the transforms: which instantiation of the analysis and
// resynthesis kernels a call runs. Host-only and header-only (no CUDA headers): the library (pv_capi.cu,
// pv_kernels.cu) and the CPU emulator (emu/pv_emu.cpp) share every rule written here.
#pragma once

#include <cstdint>
#include <string>

namespace pvk {

// Sizes served by the templated kernels of pv_body.cuh; everything else takes the generic path.
inline bool dft_size_is_templated( int N ) { return N == 256 || N == 512 || N == 1024 || N == 2048 || N == 4096 || N == 8192; }

enum class KernelKind { analysis, analysis_mirror, synthesis, synthesis_mirror, generic_analysis, generic_synthesis };

// One instantiation: the template arguments of pv_analysis_kernel<N, PT, TPS, ONE, PAD, EMIT>,
// pv_analysis_mirror_kernel<N, TPS>, pv_synthesis_kernel<N, TPS, ONE> or pv_synthesis_mirror_kernel<N, TPS, ONE, GEN>.
// PT is 16 for the mirrored kinds and 8 for the plain resynthesis. The mirrored analysis takes ONE at run time
// (AnalysisArgs::one_buffer), so it is not part of that kernel's identity. Fields a kind has no use for stay false.
struct TransformKernel
	{
	KernelKind kind = KernelKind::generic_analysis;
	int N = 0, PT = 0, TPS = 0;
	bool ONE = false, PAD = false, EMIT = false, GEN = false;

	bool operator==( const TransformKernel & o ) const
		{
		return kind == o.kind && N == o.N && PT == o.PT && TPS == o.TPS && ( ONE == o.ONE || kind == KernelKind::analysis_mirror )
		    && PAD == o.PAD && EMIT == o.EMIT && GEN == o.GEN;
		}
	bool is_analysis() const { return kind == KernelKind::analysis || kind == KernelKind::analysis_mirror || kind == KernelKind::generic_analysis; }
	// the kernel's name as a profiler shows it, normalised: pv_analysis_kernel<4096,16,512,true,false,false>
	std::string name() const
		{
		auto i = []( int v ) { return std::to_string( v ); };
		auto b = []( bool v ) { return std::string( v ? "true" : "false" ); };
		switch( kind )
			{
			case KernelKind::analysis:
				return "pv_analysis_kernel<" + i( N ) + "," + i( PT ) + "," + i( TPS ) + "," + b( ONE ) + "," + b( PAD ) + "," + b( EMIT ) + ">";
			case KernelKind::analysis_mirror: return "pv_analysis_mirror_kernel<" + i( N ) + "," + i( TPS ) + ">";
			case KernelKind::synthesis: return "pv_synthesis_kernel<" + i( N ) + "," + i( TPS ) + "," + b( ONE ) + ">";
			case KernelKind::synthesis_mirror:
				return "pv_synthesis_mirror_kernel<" + i( N ) + "," + i( TPS ) + "," + b( ONE ) + "," + b( GEN ) + ">";
			case KernelKind::generic_analysis: return "pv_generic_analysis_kernel";
			case KernelKind::generic_synthesis: return "pv_generic_synthesis_kernel";
			}
		return "";
		}
	};

// The shape of the kernels' standard form: window == dft, hop == dft/16 (every BASELINE config).
inline bool standard_shape( int N, int W, int hop ) { return W == N && hop == N / 16; }

// The analysis with the mirrored last pass (pv_body.cuh: analysis_cta_mirror) exists for dft 1024 to 4096 at the
// standard shape.
inline bool analysis_mirror_fits( int N, int W, int hop ) { return ( N == 1024 || N == 2048 || N == 4096 ) && standard_shape( N, W, hop ); }

// The mirrored resynthesis (pv_body.cuh: synthesis_cta_mirror), dft 1024 to 8192: the standard shape in its
// compile-time form, else the general form, where the window fills whole slots of the thread layout (a multiple of
// dft/16 samples) and the hop is even, at most one slot and leaves no gaps.
inline bool synthesis_mirror_fits( int N, int W, int hop )
	{
	if( !( N == 1024 || N == 2048 || N == 4096 || N == 8192 ) ) return false;
	if( standard_shape( N, W, hop ) ) return true;
	return W >= N / 16 && W % ( N / 16 ) == 0 && W <= N && hop >= 2 && hop % 2 == 0 && hop <= W && hop <= N / 16;
	}

// The 16-point one-buffer analysis takes zero-padded windows that fill whole slots (the API default shape) with vector
// loads when the input allows them.
inline bool analysis_pad_fits( const TransformKernel & k, int W, bool aligned2 )
	{
	return k.kind == KernelKind::analysis && k.PT == 16 && k.ONE && W < k.N && W % ( k.N / 16 ) == 0 && aligned2;
	}

// The full-window analysis that also leaves the phase summaries of its rows: 16 points per thread, one buffer, 512
// threads per SM, dft 2048 and up.
inline bool analysis_emit_fits( const TransformKernel & k, int W )
	{
	return k.kind == KernelKind::analysis && k.PT == 16 && k.ONE && k.TPS == 512 && k.N >= 2048 && W == k.N;
	}

// Measured on B200 (tools/experiments/exp_r1*.sh): 16 points per thread with one exchange buffer from dft 4096 up; the
// mirrored last pass for dft 1024 at the standard shape; 8 points per thread at 768 threads per SM otherwise. dft 2048
// takes 16 points per thread once the grid covers the SMs a few times over (2.52 -> 2.31 ms on a cfg4 channel), 8 for
// short signals, where twice the threads per frame matter more. That is decided on the WHOLE signal's frame count
// (`signal_frames` per channel), so that every frame-range shard of a signal runs the same arithmetic.
// aligned2: hop, W/2, the input's stride, offset and address allow 8-byte loads. emit: the caller wants the rows' phase
// summaries and their layout allows them; only the kernel that can leave them honours it.
inline TransformKernel choose_analysis( int N, int W, int hop, int C, int64_t signal_frames, int sms, bool aligned2, bool emit )
	{
	TransformKernel k;
	k.N = N;
	if( !dft_size_is_templated( N ) ) { k.kind = KernelKind::generic_analysis; return k; }
	if( N == 1024 && analysis_mirror_fits( N, W, hop ) )
		{
		k.kind = KernelKind::analysis_mirror; k.PT = 16; k.TPS = 512; k.ONE = true;
		return k;
		}
	k.kind = KernelKind::analysis;
	const bool large = (int64_t) C * signal_frames >= (int64_t) sms * 128;
	if( N >= 4096 || ( N == 2048 && large ) )
		{
		k.PT = 16; k.TPS = 512; k.ONE = true;
		k.PAD = analysis_pad_fits( k, W, aligned2 );
		k.EMIT = emit && !k.PAD && analysis_emit_fits( k, W );
		}
	else { k.PT = 8; k.TPS = 768; }
	return k;
	}

// The mirrored resynthesis wherever it fits: dft 4096 at the standard shape keeps its window and tables in tensor
// memory (128 registers, one exchange buffer, 4 CTAs per SM); dft 8192 fits two 256-thread CTAs per SM with 128
// registers and one exchange buffer (102 KB of shared memory each); the others run at 384 threads per SM. Elsewhere the
// 8-point kernel: dft 8192 with one exchange buffer and 64 registers per thread, so that two 512-thread CTAs share an SM.
inline TransformKernel choose_synthesis( int N, int W, int hop )
	{
	TransformKernel k;
	k.N = N;
	if( !dft_size_is_templated( N ) ) { k.kind = KernelKind::generic_synthesis; return k; }
	if( synthesis_mirror_fits( N, W, hop ) )
		{
		k.kind = KernelKind::synthesis_mirror; k.PT = 16;
		k.GEN = !standard_shape( N, W, hop );
		const bool wide = N == 8192 || ( N == 4096 && !k.GEN );
		k.TPS = wide ? 512 : 384; k.ONE = wide;
		return k;
		}
	k.kind = KernelKind::synthesis; k.PT = 8;
	k.TPS = N == 8192 ? 1024 : 768; k.ONE = N == 8192;
	return k;
	}

} // namespace pvk
