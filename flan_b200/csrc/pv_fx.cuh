// flan_b200/csrc/pv_fx.cuh
//
// Expression programs: a Function<TF, float> written as a small expression of t and f (flan/fx.h) instead of a lambda,
// encoded as postfix ops over a value stack (flan_b200_fx_program, include/flan_b200.h). The library knows what such a
// program depends on, samples it on the device (pv_fx.cu) and evaluates it on the host (flan_b200_fx_eval) with the
// same source: fx_eval is PVM_HD like interp_eval, and both translation units that compile it do so without FMA
// contraction (nvcc -fmad=false for pv_fx.cu, -ffp-contract=off for the host side). Every node is one IEEE float32
// operation with round to nearest, in the order the user wrote the tree; nothing is folded or reassociated. The five
// transcendental ops compute (float) fn( (double) x ), as interpolators 7 and 8 do: there CUDA's and glibc's double
// results may round to different floats near a tie, the only place the two sides can differ.
#pragma once

#include "../../include/flan_b200.h"
#include "pv_modify_body.cuh"      // PVM_HD, interp_eval

namespace pvfx {

using Program = flan_b200_fx_program;

// fminf / fmaxf: a NaN operand yields the other operand; of two zeros, min picks -0 and max +0 (IEEE leaves that choice
// open, and the two sides must agree).
PVM_HD bool fx_neg_zero( float a ) { return a == 0.0f && 1.0f / a < 0.0f; }
PVM_HD float fx_min( float a, float b )
	{
	if( a != a ) return b;
	if( b != b ) return a;
	if( a == b ) return fx_neg_zero( a ) ? a : b;
	return a < b ? a : b;
	}
PVM_HD float fx_max( float a, float b )
	{
	if( a != a ) return b;
	if( b != b ) return a;
	if( a == b ) return fx_neg_zero( a ) ? b : a;
	return a < b ? b : a;
	}

// Breakpoint envelope: x <= x_0 -> y_0, x >= x_n -> y_n, NaN -> NaN, else y_i + interp( u ) * ( y_{i+1} - y_i ) with
// u = ( x - x_i ) / ( x_{i+1} - x_i ) and x_i <= x < x_{i+1}.
PVM_HD float fx_curve( const flan_b200_fx_curve & c, float x )
	{
	if( x != x ) return x;
	const int n = c.points;
	if( x <= c.x[0] ) return c.y[0];
	if( x >= c.x[n - 1] ) return c.y[n - 1];
	int i = 0;
	while( i + 2 < n && c.x[i + 1] <= x ) ++i;
	const float u = ( x - c.x[i] ) / ( c.x[i + 1] - c.x[i] );
	return c.y[i] + pvm::interp_eval( c.interp, u ) * ( c.y[i + 1] - c.y[i] );
	}

// The one NaN a program returns, 0x7fc00000 on both sides: CUDA's arithmetic makes 0x7fffffff and x86's 0xffc00000, and
// a table sampled on the device must hold the bits the host evaluation of the same program gives.
PVM_HD float fx_canonical( float v )
	{
	if( v == v ) return v;
#if defined( __CUDA_ARCH__ )
	return __int_as_float( 0x7fc00000 );
#else
	const uint32_t bits = 0x7fc00000u;
	float q;
	__builtin_memcpy( &q, &bits, 4 );
	return q;
#endif
	}

// Evaluates a program that fx_check accepted. NaN payloads never change a non-NaN result (comparisons, WHERE, MIN / MAX
// and CURVE only test for NaN), so canonicalising the result alone makes both sides agree bit for bit.
PVM_HD float fx_eval( const Program & p, float t, float f )
	{
	float s[FLAN_B200_FX_MAX_STACK];
	int sp = 0;
	for( int k = 0; k < p.ops; ++k )
		{
		const flan_b200_fx_op o = p.op[k];
		float r;
		switch( o.code )
			{
			case FLAN_B200_FX_T: s[sp++] = t; continue;
			case FLAN_B200_FX_F: s[sp++] = f; continue;
			case FLAN_B200_FX_CONST: s[sp++] = o.value; continue;
			default: break;
			}
		const float a = s[sp - 1];
		switch( o.code )      // one operand
			{
			case FLAN_B200_FX_NEG: s[sp - 1] = -a; continue;
			case FLAN_B200_FX_ABS: s[sp - 1] = fabsf( a ); continue;
			case FLAN_B200_FX_FLOOR: s[sp - 1] = floorf( a ); continue;
			case FLAN_B200_FX_CEIL: s[sp - 1] = ceilf( a ); continue;
			case FLAN_B200_FX_ROUND: s[sp - 1] = roundf( a ); continue;
			case FLAN_B200_FX_SQRT: s[sp - 1] = sqrtf( a ); continue;
			case FLAN_B200_FX_SIN: s[sp - 1] = (float) sin( (double) a ); continue;
			case FLAN_B200_FX_COS: s[sp - 1] = (float) cos( (double) a ); continue;
			case FLAN_B200_FX_EXP: s[sp - 1] = (float) exp( (double) a ); continue;
			case FLAN_B200_FX_LOG: s[sp - 1] = (float) log( (double) a ); continue;
			case FLAN_B200_FX_CURVE: s[sp - 1] = fx_curve( p.curve[o.index], a ); continue;
			default: break;
			}
		if( o.code == FLAN_B200_FX_WHERE )     // c a b -> c != 0 ? a : b
			{
			sp -= 2;
			s[sp - 1] = s[sp - 1] != 0.0f ? s[sp] : s[sp + 1];
			continue;
			}
		const float x = s[sp - 2];      // two operands: x op a
		switch( o.code )
			{
			case FLAN_B200_FX_ADD: r = x + a; break;
			case FLAN_B200_FX_SUB: r = x - a; break;
			case FLAN_B200_FX_MUL: r = x * a; break;
			case FLAN_B200_FX_DIV: r = x / a; break;
			case FLAN_B200_FX_MIN: r = fx_min( x, a ); break;
			case FLAN_B200_FX_MAX: r = fx_max( x, a ); break;
			case FLAN_B200_FX_LT: r = x < a ? 1.0f : 0.0f; break;
			case FLAN_B200_FX_LE: r = x <= a ? 1.0f : 0.0f; break;
			case FLAN_B200_FX_GT: r = x > a ? 1.0f : 0.0f; break;
			case FLAN_B200_FX_GE: r = x >= a ? 1.0f : 0.0f; break;
			case FLAN_B200_FX_EQ: r = x == a ? 1.0f : 0.0f; break;
			case FLAN_B200_FX_NE: r = x != a ? 1.0f : 0.0f; break;
			default: r = (float) pow( (double) x, (double) a ); break;       // FLAN_B200_FX_POW
			}
		s[--sp - 1] = r;
		}
	return fx_canonical( s[0] );
	}

} // namespace pvfx
