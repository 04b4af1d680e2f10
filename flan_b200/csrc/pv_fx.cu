// flan_b200/csrc/pv_fx.cu -- sm_100a kernels of the expression Functions (pv_fx.cuh): the grid sampler behind
// PV::repitch / stretch / modify_time / modify_frequency and the evaluation at every MF behind PV::modify_frequency.
// Compiled with -fmad=false: fx_eval's float nodes are the host's bit for bit. The program travels by value as a kernel
// parameter (__grid_constant__: read from the parameter bank, never copied), so concurrent calls on one context share
// nothing. Each thread writes one float per value; the interpreter's stack lives in local memory (DESIGN §4.6).
#include "pv_fx.h"

namespace pvfx {

// Value i of the view: x = i / B, y = i % B (t and f), x = i (t alone), y = i (f alone), nothing (neither).
__global__ void __launch_bounds__( 256 ) pv_fx_sample_kernel( const __grid_constant__ Program p, int64_t total, int B, int uses_t, int uses_f,
                                                              float time_step, float bin_width, float * out )
	{
	for( int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t) gridDim.x * blockDim.x )
		{
		const int64_t x = uses_t ? ( uses_f ? i / B : i ) : 0;
		const int64_t y = uses_f ? ( uses_t ? i % B : i ) : 0;
		out[i] = fx_eval( p, float( x ) * time_step, float( y ) * bin_width );
		}
	}

// out[c][x][b] = program( float( x ) / frame_rate, pv[c][x][b].f ).
__global__ void __launch_bounds__( 256 ) pv_fx_at_pv_kernel( const __grid_constant__ Program p, const float2 * pv, int64_t total, int64_t F, int B,
                                                             float frame_rate, float * out )
	{
	for( int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t) gridDim.x * blockDim.x )
		{
		const int64_t x = ( i / B ) % F;
		out[i] = fx_eval( p, float( x ) / frame_rate, pv[i].y );
		}
	}

namespace {
unsigned grid_for( int64_t total, int sms )
	{
	const int64_t blocks = ( total + 255 ) / 256, cap = (int64_t) sms * 8;
	return (unsigned)( blocks < cap ? ( blocks < 1 ? 1 : blocks ) : cap );
	}
}

cudaError_t launch_fx_sample( const Program & p, int64_t total, int B, bool uses_t, bool uses_f, float time_step, float bin_width,
                              float * out, int sms, cudaStream_t st )
	{
	pv_fx_sample_kernel<<<grid_for( total, sms ), 256, 0, st>>>( p, total, B, uses_t, uses_f, time_step, bin_width, out );
	return cudaGetLastError();
	}

cudaError_t launch_fx_at_pv( const Program & p, const float * pv, int64_t total, int64_t F, int B, float frame_rate, float * out,
                             int sms, cudaStream_t st )
	{
	pv_fx_at_pv_kernel<<<grid_for( total, sms ), 256, 0, st>>>( p, (const float2 *) pv, total, F, B, frame_rate, out );
	return cudaGetLastError();
	}

} // namespace pvfx
