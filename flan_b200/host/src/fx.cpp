// flan::fx (flan/fx.h): expressions are built by concatenating postfix programs (include/flan_b200.h,
// flan_b200_fx_program) and checked by the library as they grow, so an Expr is either a program the GPU accepts or
// carries the reason it is not.
#include "flan/fx.h"

#include <limits>

#include "flan/Utility/Interpolator.h"
#include "flan_b200.h"

namespace flan::fx {

namespace {

using Program = flan_b200_fx_program;

const std::string too_long = "fx: expression of more than " + std::to_string( FLAN_B200_FX_MAX_OPS ) + " ops or "
                             + std::to_string( FLAN_B200_FX_MAX_CURVES ) + " curves";

// Appends src's ops to dst, src's curves after dst's (their op indices shifted to match). False when a limit is passed.
bool append( Program & dst, const Program & src )
	{
	if( dst.ops + src.ops > FLAN_B200_FX_MAX_OPS || dst.curves + src.curves > FLAN_B200_FX_MAX_CURVES ) return false;
	for( int i = 0; i < src.ops; ++i )
		{
		flan_b200_fx_op o = src.op[i];
		if( o.code == FLAN_B200_FX_CURVE ) o.index += dst.curves;
		dst.op[dst.ops++] = o;
		}
	for( int c = 0; c < src.curves; ++c ) dst.curve[dst.curves++] = src.curve[c];
	return true;
	}

}

Expr Expr::invalid( const std::string & why )
	{
	Expr e;
	e.error_ = why;
	return e;
	}

Expr Expr::leaf( int code )
	{
	auto p = std::make_shared<Program>();
	p->ops = 1;
	p->op[0] = flan_b200_fx_op{ code, 0, 0.0f };
	Expr e;
	e.program_ = std::move( p );
	return e;
	}

Expr::Expr( float constant ) : Expr( leaf( FLAN_B200_FX_CONST ) )
	{
	std::const_pointer_cast<Program>( program_ )->op[0].value = constant;
	}

Expr Expr::apply( int code, std::initializer_list<const Expr *> operands )
	{
	auto p = std::make_shared<Program>();
	for( const Expr * a : operands )
		{
		if( !a->valid() ) return *a;
		if( !append( *p, *a->program() ) ) return invalid( too_long );
		}
	if( p->ops == FLAN_B200_FX_MAX_OPS ) return invalid( too_long );
	p->op[p->ops++] = flan_b200_fx_op{ code, 0, 0.0f };
	if( flan_b200_fx_check( p.get(), nullptr, nullptr ) != FLAN_B200_OK ) return invalid( std::string( "fx: " ) + flan_b200_fx_last_error() );
	Expr e;
	e.program_ = std::move( p );
	return e;
	}

float Expr::operator()( TF x ) const
	{
	float out = std::numeric_limits<float>::quiet_NaN();
	if( valid() ) flan_b200_fx_eval( program_.get(), x.t, x.f, &out );
	return out;
	}

const Expr t = Expr::leaf( FLAN_B200_FX_T );
const Expr f = Expr::leaf( FLAN_B200_FX_F );

Expr operator+( const Expr & a, const Expr & b ) { return Expr::apply( FLAN_B200_FX_ADD, { &a, &b } ); }
Expr operator-( const Expr & a, const Expr & b ) { return Expr::apply( FLAN_B200_FX_SUB, { &a, &b } ); }
Expr operator*( const Expr & a, const Expr & b ) { return Expr::apply( FLAN_B200_FX_MUL, { &a, &b } ); }
Expr operator/( const Expr & a, const Expr & b ) { return Expr::apply( FLAN_B200_FX_DIV, { &a, &b } ); }
Expr operator-( const Expr & a ) { return Expr::apply( FLAN_B200_FX_NEG, { &a } ); }
Expr operator<( const Expr & a, const Expr & b ) { return Expr::apply( FLAN_B200_FX_LT, { &a, &b } ); }
Expr operator<=( const Expr & a, const Expr & b ) { return Expr::apply( FLAN_B200_FX_LE, { &a, &b } ); }
Expr operator>( const Expr & a, const Expr & b ) { return Expr::apply( FLAN_B200_FX_GT, { &a, &b } ); }
Expr operator>=( const Expr & a, const Expr & b ) { return Expr::apply( FLAN_B200_FX_GE, { &a, &b } ); }
Expr operator==( const Expr & a, const Expr & b ) { return Expr::apply( FLAN_B200_FX_EQ, { &a, &b } ); }
Expr operator!=( const Expr & a, const Expr & b ) { return Expr::apply( FLAN_B200_FX_NE, { &a, &b } ); }
Expr abs( const Expr & a ) { return Expr::apply( FLAN_B200_FX_ABS, { &a } ); }
Expr floor( const Expr & a ) { return Expr::apply( FLAN_B200_FX_FLOOR, { &a } ); }
Expr ceil( const Expr & a ) { return Expr::apply( FLAN_B200_FX_CEIL, { &a } ); }
Expr round( const Expr & a ) { return Expr::apply( FLAN_B200_FX_ROUND, { &a } ); }
Expr sqrt( const Expr & a ) { return Expr::apply( FLAN_B200_FX_SQRT, { &a } ); }
Expr min( const Expr & a, const Expr & b ) { return Expr::apply( FLAN_B200_FX_MIN, { &a, &b } ); }
Expr max( const Expr & a, const Expr & b ) { return Expr::apply( FLAN_B200_FX_MAX, { &a, &b } ); }
Expr where( const Expr & c, const Expr & a, const Expr & b ) { return Expr::apply( FLAN_B200_FX_WHERE, { &c, &a, &b } ); }
Expr sin( const Expr & a ) { return Expr::apply( FLAN_B200_FX_SIN, { &a } ); }
Expr cos( const Expr & a ) { return Expr::apply( FLAN_B200_FX_COS, { &a } ); }
Expr exp( const Expr & a ) { return Expr::apply( FLAN_B200_FX_EXP, { &a } ); }
Expr log( const Expr & a ) { return Expr::apply( FLAN_B200_FX_LOG, { &a } ); }
Expr pow( const Expr & a, const Expr & b ) { return Expr::apply( FLAN_B200_FX_POW, { &a, &b } ); }

Expr curve( const Expr & x, std::initializer_list<Expr::Point> points, const Interpolator & interp )
	{
	if( interp.get_device_id() < 0 ) return Expr::invalid( "fx::curve: only the named Interpolators (linear ... sqrt) have a GPU form" );
	if( points.size() < 1 || points.size() > FLAN_B200_FX_MAX_POINTS )
		return Expr::invalid( "fx::curve: needs 1 to " + std::to_string( FLAN_B200_FX_MAX_POINTS ) + " points" );
	if( !x.valid() ) return x;
	auto p = std::make_shared<Program>( *x.program() );
	if( p->ops == FLAN_B200_FX_MAX_OPS || p->curves == FLAN_B200_FX_MAX_CURVES ) return Expr::invalid( too_long );
	flan_b200_fx_curve & c = p->curve[p->curves];
	c.points = int( points.size() );
	c.interp = interp.get_device_id();
	int i = 0;
	for( const Expr::Point & q : points ) { c.x[i] = q.x; c.y[i] = q.y; ++i; }
	p->op[p->ops++] = flan_b200_fx_op{ FLAN_B200_FX_CURVE, p->curves++, 0.0f };
	if( flan_b200_fx_check( p.get(), nullptr, nullptr ) != FLAN_B200_OK ) return Expr::invalid( std::string( "fx::curve: " ) + flan_b200_fx_last_error() );
	Expr e;
	e.program_ = std::move( p );
	return e;
	}

}
