// flan::Function of the B200 build: the argument type of the PV-domain methods (reference src/flan/Function.h:35-103),
// restated for what this build needs of it -- a constant or a callable, plus the execution policy the reference
// carries along for sampling user lambdas on the host (Utility/execution.h:20-26) -- and, for Function<TF, float>, an
// expression of t and f (flan/fx.h) that the PV-domain methods sample on the GPU.
#pragma once

#include <concepts>
#include <functional>
#include <type_traits>
#include <variant>

#include "flan/defines.h"
#include "flan/fx.h"

namespace flan {

enum class ExecutionPolicy { Linear_Sequenced, Linear_Unsequenced, Parallel_Sequenced, Parallel_Unsequenced };

template<typename I, typename O>
struct Function
	{
	using StdFuncType = std::function<O( I )>;
	using ReturnType = O;
	using ArgType = I;

	Function( const Function & ) = delete;
	Function & operator=( const Function & ) = delete;
	Function( Function && ) = default;
	Function & operator=( Function && ) = default;

	/** A constant: `pv.repitch( 1.5f )`. */
	template<typename T> requires std::convertible_to<T, O>
	Function( T constant ) : f( static_cast<O>( constant ) ), execution_policy( ExecutionPolicy::Parallel_Unsequenced ) {}

	/** Anything callable as O( I ): `pv.repitch( []( TF tf ){ return tf.t; } )`. */
	template<typename T> requires ( std::convertible_to<T, StdFuncType> && !std::convertible_to<T, O>
	                                && !std::same_as<std::remove_cvref_t<T>, fx::Expr> )
	Function( T && callable, ExecutionPolicy policy = ExecutionPolicy::Parallel_Unsequenced )
		: f( StdFuncType( std::forward<T>( callable ) ) ), execution_policy( policy ) {}

	/** An expression of t and f: `pv.stretch( 1.0f + fx::t / 20.0f )`. */
	Function( fx::Expr expr ) requires ( std::same_as<I, TF> && std::same_as<O, float> )
		: f( std::move( expr ) ), execution_policy( ExecutionPolicy::Parallel_Unsequenced ) {}

	Function copy() const
		{
		if( is_constant() ) return Function( std::get<O>( f ) );
		if constexpr ( std::same_as<I, TF> && std::same_as<O, float> )
			if( const fx::Expr * e = expr() ) return Function( *e );
		return Function( std::get<StdFuncType>( f ), execution_policy );
		}

	bool is_constant() const { return std::holds_alternative<O>( f ); }
	/** The expression this Function holds, or null. */
	const fx::Expr * expr() const { return std::get_if<fx::Expr>( &f ); }
	ExecutionPolicy get_execution_policy() const { return execution_policy; }

	O operator()( I x ) const
		{
		if( is_constant() ) return std::get<O>( f );
		if constexpr ( std::same_as<I, TF> && std::same_as<O, float> )
			if( const fx::Expr * e = expr() ) return ( *e )( x );
		return std::get<StdFuncType>( f )( x );
		}

private:
	std::variant<O, StdFuncType, fx::Expr> f;
	ExecutionPolicy execution_policy;
	};

}
