// flan::PV of the B200 build: the conversion entry points of the reference's PV (src/flan/PV/PV.h:27-490) on the
// phase-vocoder path, with the reference's signatures (PV.h:88-96), and the PV-domain methods that BASELINE config 4
// chains between them (PV.h:276-308).
#pragma once

#include "flan/PV/PVBuffer.h"
#include "flan/Function.h"
#include "flan/Utility/Interpolator.h"

namespace flan {

class Audio;

class PV : public PVBuffer
{
public:
	PV() : PVBuffer( PVBuffer::Format() ) {}
	PV( PVBuffer && other ) : PVBuffer( std::move( other ) ) {}

	static PV create_null() { return PVBuffer(); }

	/** Phase accumulation, inverse FFT and windowed overlap-add (reference Conversions/AudioPV.cpp:86-139), on the GPU.
	 *  A NaN/Inf in the data prints the reference's warning and conversion continues (AudioPV.cpp:88-89). */
	Audio convert_to_audio( flan_CANCEL_ARG ) const;

	/** convert_to_audio() then convert_to_left_right(); null unless stereo (AudioPV.cpp:141-145). */
	Audio convert_to_lr_audio( flan_CANCEL_ARG ) const;

	// ---- PV-domain chain (reference PV/PVModify.cpp:196-385), on the GPU, data stays device-resident -------------
	// A lambda Function argument is sampled over the frame x bin grid on the host, as the reference does (PV.h:31-35); a
	// constant Function is passed to the device as a single value. An expression of t and f (flan/fx.h, e.g.
	// `1.0f + fx::t / 20.0f`) is sampled on the GPU into the table its dependence needs -- one value, one per frame, one
	// per bin, or the grid -- so a time-only stretch / modify_time and a frequency-only repitch take the kernels a
	// constant takes, modify_frequency evaluates it at every MF on the device without downloading the PV, and on a sharded
	// PV a time-only stretch / modify_time keeps the shards. Same results as the lambda [&]( TF x ){ return e( x ); }.
	// An invalid expression (past its limits, or a curve with a user-callable Interpolator) prints why and yields a null
	// PV. NOTE: in the reference a constant Function makes
	// repitch / stretch alias one scalar (FunctionSample.h:185-189: `at( f, b ) += at( f, b - 1 )` doubles it every
	// step until it overflows), which is undefined further down (float -> int of inf, PVModify.cpp:222,312-315); here
	// a constant behaves like the lambda that returns it -- the evident intent. Named interpolators only
	// (Interpolator::linear() ... ::sqrt()); a user callable has no device form and yields a null PV with a message.

	/** Frequency mapping: \param mod takes time/frequency pairs and returns frequency (PV.h:276-283). */
	PV modify_frequency( const Function<TF, Frequency> & mod, const Interpolator & = Interpolator::linear() ) const;

	/** Time mapping: \param mod takes time/frequency pairs and returns time (PV.h:285-292). */
	PV modify_time( const Function<TF, Second> & mod, const Interpolator & = Interpolator::linear() ) const;

	/** \param factor takes time/frequency pairs and returns a frequency multiplier (PV.h:294-301). */
	PV repitch( const Function<TF, float> & factor, const Interpolator & = Interpolator::linear() ) const;

	/** \param factor takes time/frequency pairs and returns a time multiplier (PV.h:303-310). */
	PV stretch( const Function<TF, float> & factor, const Interpolator & = Interpolator::linear() ) const;
};

}
