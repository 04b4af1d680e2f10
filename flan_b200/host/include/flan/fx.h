// flan::fx -- expression Functions of the B200 build. A Function<TF, float> written as an expression of the time t and
// the frequency f instead of a lambda:
//     pv.stretch( 1.0f + fx::t / 20.0f );
//     pv.repitch( fx::curve( fx::t, { { 0, 1 }, { 2, 1.5f } }, Interpolator::smoothstep() ) );
// The library knows what such an expression depends on, so the PV-domain methods sample it on the GPU into the smallest
// table it needs -- one value, one per frame, one per bin, or the whole grid -- and a time-only stretch or a
// frequency-only repitch takes the same kernels a constant does. Evaluated on the host (operator()), it runs the very
// code the GPU runs (flan_b200_fx_eval, include/flan_b200.h): float32 nodes in the order written, nothing folded or
// reassociated; sin, cos, exp, log and pow are computed in double and rounded.
//
// Limits: 64 ops, a stack of 16 values, 8 curves of at most 64 points (strictly ascending x, named Interpolators only).
// An expression past them, or a curve with a user-callable Interpolator, is invalid: its error() says why, the
// PV-domain methods print it and return a null PV, and operator() returns NaN.
#pragma once

#include <initializer_list>
#include <memory>
#include <string>

#include "flan/defines.h"

struct flan_b200_fx_program;

namespace flan {

struct Interpolator;

namespace fx {

class Expr
	{
public:
	Expr( float constant );

	/** The expression at one point, evaluated by the library's host evaluator (NaN for an invalid expression). */
	float operator()( TF x ) const;

	bool valid() const { return error_.empty(); }
	const std::string & error() const { return error_; }
	/** The encoded program (include/flan_b200.h), or null when invalid. */
	const flan_b200_fx_program * program() const { return error_.empty() ? program_.get() : nullptr; }

	// building blocks of the operators and functions below (op codes FLAN_B200_FX_*): a push, an op over its operands'
	// programs in order, and an invalid expression
	static Expr leaf( int code );
	static Expr apply( int code, std::initializer_list<const Expr *> operands );
	static Expr invalid( const std::string & why );

	struct Point { float x, y; };
	friend Expr curve( const Expr & x, std::initializer_list<Point> points, const Interpolator & interp );

private:
	Expr() = default;
	std::shared_ptr<const flan_b200_fx_program> program_;
	std::string error_;
	};

/** The placeholders: time in seconds and frequency in Hz of the point being evaluated. */
extern const Expr t;
extern const Expr f;

Expr operator+( const Expr & a, const Expr & b );
Expr operator-( const Expr & a, const Expr & b );
Expr operator*( const Expr & a, const Expr & b );
Expr operator/( const Expr & a, const Expr & b );
Expr operator-( const Expr & a );
/** Comparisons give 1.0f or 0.0f. */
Expr operator<( const Expr & a, const Expr & b );
Expr operator<=( const Expr & a, const Expr & b );
Expr operator>( const Expr & a, const Expr & b );
Expr operator>=( const Expr & a, const Expr & b );
Expr operator==( const Expr & a, const Expr & b );
Expr operator!=( const Expr & a, const Expr & b );

Expr abs( const Expr & a );
Expr floor( const Expr & a );
Expr ceil( const Expr & a );
/** Half away from zero (roundf). */
Expr round( const Expr & a );
Expr sqrt( const Expr & a );
/** fminf / fmaxf: a NaN operand yields the other one; -0 counts as less than +0. */
Expr min( const Expr & a, const Expr & b );
Expr max( const Expr & a, const Expr & b );
/** c != 0 ? a : b (both sides evaluated). */
Expr where( const Expr & c, const Expr & a, const Expr & b );
Expr sin( const Expr & a );
Expr cos( const Expr & a );
Expr exp( const Expr & a );
Expr log( const Expr & a );
Expr pow( const Expr & a, const Expr & b );
/** Breakpoint envelope over strictly ascending x: y_0 at and before the first point, y_n at and after the last, and
 *  y_i + interp( u ) * ( y_{i+1} - y_i ), u = ( x - x_i ) / ( x_{i+1} - x_i ), in between. */
Expr curve( const Expr & x, std::initializer_list<Expr::Point> points, const Interpolator & interp );

}
}
