// The four conversion entry points of the phase-vocoder path in the B200 build. Signatures, defaults and error
// behaviour are the reference's (src/flan/Conversions/AudioPV.cpp:12-145); the bodies call the C ABI of
// libflan_b200.so (include/flan_b200.h) on device-resident storage instead of FFTW plans and per-frame CPU loops.
#include "flan/Audio/Audio.h"
#include "flan/PV/PV.h"

#include <functional>
#include <iostream>

#include "flan_b200.h"

namespace flan {

Audio::Audio() : AudioBuffer() {}
Audio::Audio( AudioBuffer && other ) : AudioBuffer( std::move( other ) ) {}
Audio Audio::copy() const { return AudioBuffer::copy(); }

Audio Audio::create_null()
	{
	std::cout << "Null Audio created";          // AudioConstructors.cpp:19-23
	return Audio();
	}

Audio Audio::create_from_buffer( std::vector<float> && buffer, Channel num_channels, FrameRate sr )
	{
	return AudioBuffer( std::move( buffer ), num_channels, sr );
	}

Audio Audio::create_from_format( const AudioBuffer::Format & f ) { return AudioBuffer( f ); }

namespace {

// Below this much PV data one GPU finishes before several could be fed (a 10 s stereo signal at dft 2048 is 56 MB).
constexpr size_t MULTI_MIN_PV_BYTES = size_t( 256 ) << 20;

// std::atomic<bool> canceller -> the plain int flag the C ABI polls on entry and between the slices of its pipelined
// forms. The calls only ENQUEUE GPU work (microseconds), so the protocol of flan_CANCEL_POINT (defines.h:52-62) is kept
// by checking the canceller before the call and again before the result object is handed out; work already enqueued is
// not recalled, its result is dropped.
struct CancelFlag
	{
	volatile int value;
	explicit CancelFlag( std::atomic<bool> & c ) : value( c.load() ? 1 : 0 ) {}
	};

int report( flan_b200_ctx * ctx, const char * what, int rc )
	{
	if( rc != FLAN_B200_OK && rc != FLAN_B200_CANCELLED )
		std::cout << "flan::" << what << " failed on the GPU engine: " << flan_b200_last_error( ctx ) << std::endl;
	return rc;
	}

}

PV Audio::convert_to_PV( Frame window_size, Frame hop, Frame dft_size, flan_CANCEL_ARG_CPP ) const
	{
	flan_CANCEL_POINT( PV() );
	flan_b200_ctx * ctx = b200::context();
	if( !ctx || hop < 1 ) return PV();

	PVBuffer::Format f;                                                  // AudioPV.cpp:20-26
	f.num_channels = get_num_channels();
	f.num_frames = Frame( flan_b200_num_frames( get_num_frames(), hop ) );
	f.num_bins = dft_size / 2 + 1;
	f.sample_rate = get_sample_rate();
	f.analysis_rate = flan_b200_analysis_rate( get_sample_rate(), hop );
	f.window_size = window_size;
	if( f.num_channels < 1 ) return PV( PVBuffer( f ) );

	// Several GPUs and a long signal whose newest copy is the host vector: frame-range shards, one per device, each
	// uploaded with its halo and analysed where it lands (no exchange); the PV stays sharded on the devices.
	if( flan_b200_multi * m = b200::multi() )
		if( const Sample * h = storage().host_data_if_current() )
			{
			const size_t pv_bytes = sizeof( MF ) * size_t( f.num_channels ) * size_t( f.num_frames ) * size_t( f.num_bins );
			int shards = 1; int64_t begin[FLAN_B200_MAX_DEVICES + 1];
			if( pv_bytes >= MULTI_MIN_PV_BYTES
			 && flan_b200_multi_plan( m, f.num_channels, get_num_frames(), window_size, hop, dft_size, &shards, begin ) == FLAN_B200_OK && shards > 1 )
				{
				auto store = b200::new_sharded_store();
				auto * desc = static_cast<flan_b200_sharded_pv *>( b200::sharded_descriptor( *store ) );
				if( flan_b200_multi_convert_to_pv_host( m, h, f.num_channels, get_num_frames(), get_sample_rate(), window_size, hop, dft_size, desc ) != FLAN_B200_OK )
					{
					std::cout << "flan::Audio::convert_to_PV failed on the GPU engine: " << flan_b200_multi_last_error( m ) << std::endl;
					return PV();
					}
				if( canceller ) return PV();
				return PV( PVBuffer::from_device_result( f, b200::Mirror<MF>::from_shards( pv_bytes / sizeof( MF ), std::move( store ) ) ) );
				}
			}

	MF * d_pv = nullptr;
	b200::Mirror<MF> data = b200::Mirror<MF>::device_result( size_t( f.num_channels ) * size_t( f.num_frames ) * size_t( f.num_bins ), &d_pv );
	if( !d_pv ) return PV();

	CancelFlag cancel( canceller );
	const Frame n = get_num_frames();
	const Channel C = f.num_channels;
	const FrameRate sr = get_sample_rate();
	// When the newest copy of the samples is the host vector, the upload is pipelined with the transform: the engine
	// copies the samples in a few slices and analyses each slice's frames as soon as they have arrived.
	int up_rc = FLAN_B200_OK;
	const std::function<int( const Sample *, Sample * )> pipelined = [&]( const Sample * h, Sample * d )
		{
		up_rc = flan_b200_convert_to_pv_h2d( ctx, h, d, C, n, sr, window_size, hop, dft_size, reinterpret_cast<float *>( d_pv ), &cancel.value );
		return up_rc;
		};
	bool transformed = false;
	const Sample * d_audio = storage().device_with( &pipelined, &transformed );
	if( !d_audio )
		{
		if( up_rc != FLAN_B200_OK ) report( ctx, "Audio::convert_to_PV", up_rc );
		return PV();
		}
	const int rc = transformed ? FLAN_B200_OK : report( ctx, "Audio::convert_to_PV", flan_b200_convert_to_pv( ctx, d_audio, C, n,
		sr, window_size, hop, dft_size, reinterpret_cast<float *>( d_pv ), &cancel.value ) );
	if( rc != FLAN_B200_OK || canceller ) return PV();
	return PV( PVBuffer::from_device_result( f, std::move( data ) ) );
	}

PV Audio::convert_to_ms_PV( Frame window_size, Frame hop, Frame dft_size, flan_CANCEL_ARG_CPP ) const
	{
	if( get_num_channels() != 2 ) return PV();                           // AudioPV.cpp:82
	return convert_to_mid_side().convert_to_PV( window_size, hop, dft_size, canceller );
	}

Audio Audio::convert_to_mid_side() const
	{
	if( is_null() ) return Audio::create_null();                         // AudioConversions.cpp:34
	if( get_num_channels() != 2 )
		{
		std::cout << "Can't transform non-stereo Audio between Mid-Side and Left-Right formats." << std::endl;
		return copy();                                                   // AudioConversions.cpp:36-40
		}
	flan_b200_ctx * ctx = b200::context();
	if( !ctx ) return Audio::create_null();
	const Sample * d_in = storage().device();
	Sample * d_out = nullptr;
	b200::Mirror<Sample> data = b200::Mirror<Sample>::device_result( storage().size(), &d_out );
	if( !d_in || !d_out ) return Audio::create_null();
	if( report( ctx, "Audio::convert_to_mid_side", flan_b200_mid_side( ctx, d_in, d_out, get_num_frames() ) ) != FLAN_B200_OK )
		return Audio::create_null();
	return Audio( AudioBuffer::from_device_result( get_format(), std::move( data ) ) );
	}

Audio Audio::convert_to_left_right() const
	{
	return convert_to_mid_side();                                        // AudioConversions.cpp:53-56
	}

Audio PV::convert_to_audio( flan_CANCEL_ARG_CPP ) const
	{
	flan_CANCEL_POINT( Audio::create_null() );
	flan_b200_ctx * ctx = b200::context();
	if( !ctx ) return Audio::create_null();

	AudioBuffer::Format af;                                              // AudioPV.cpp:91-94
	af.num_channels = get_num_channels();
	af.num_frames = get_num_frames() * get_hop_size();
	af.sample_rate = get_sample_rate();
	if( storage().empty() ) return Audio( AudioBuffer( af ) );

	// A PV sharded over several GPUs: every device resynthesises its frames (phase state and overlap-add halo exchanged
	// device to device) and copies the samples it owns straight into the result's host vector.
	if( const auto & store = storage().shards() )
		if( flan_b200_multi * m = b200::multi() )
			{
			bool pinned = false;
			std::vector<Sample> host = b200::pool_take<Sample>( size_t( af.num_channels ) * size_t( af.num_frames ), false, &pinned );
			int nan_or_inf = 0;
			const auto * desc = static_cast<const flan_b200_sharded_pv *>( b200::sharded_descriptor( *store ) );
			// shards still exactly as PV::stretch / modify_time wrote them: the phase summaries it left are used
			if( b200::sharded_summaries( *store ) ) flan_b200_multi_promise_unchanged( m, desc );
			const int rc = flan_b200_multi_convert_to_audio_host( m, desc, host.data(), &nan_or_inf );
			if( rc != FLAN_B200_OK )
				{
				std::cout << "flan::PV::convert_to_audio failed on the GPU engine: " << flan_b200_multi_last_error( m ) << std::endl;
				return Audio::create_null();
				}
			if( nan_or_inf )                                                 // AudioPV.cpp:88-89: warn and carry on
				std::cout << "flan::convert_to_audio recieved a nan or infinite value. This often happens when dividing by zero in an earlier algorithm.";
			if( canceller ) return Audio::create_null();
			return Audio( AudioBuffer::from_device_result( af, b200::Mirror<Sample>::adopt_host( std::move( host ), pinned ) ) );
			}

	const MF * d_pv = storage().device();
	Sample * d_audio = nullptr, * h_audio = nullptr;
	b200::Mirror<Sample> data = b200::Mirror<Sample>::device_result( size_t( af.num_channels ) * size_t( af.num_frames ), &d_audio, &h_audio );
	if( !d_pv || !d_audio ) return Audio::create_null();

	CancelFlag cancel( canceller );
	// No stream-wide synchronise here: the is_nan_or_inf() pre-scan of AudioPV.cpp:88 runs on the device with the phase
	// summaries, and its warning is printed by the first host access of the result (b200_storage.cpp: sync_to_host).
	// When a recycled page-locked vector is at hand, the engine also copies the samples to the host slice by slice behind
	// the transform, so a later get_buffer() only waits for the tail of that copy.
	int rc;
	// rows that are still exactly what their producer wrote: phase summaries it left behind (PV::stretch) are used
	if( storage().device_untouched() ) flan_b200_promise_unchanged( ctx, reinterpret_cast<const float *>( d_pv ) );
	if( h_audio )
		{
		const volatile int * flag = nullptr;
		rc = report( ctx, "PV::convert_to_audio", flan_b200_convert_to_audio_d2h( ctx, reinterpret_cast<const float *>( d_pv ),
			get_num_channels(), get_num_frames(), get_num_bins(), get_sample_rate(), get_analysis_rate(), get_window_size(),
			d_audio, h_audio, &cancel.value, &flag ) );
		data.set_nan_flag( flag );
		}
	else
		{
		int nan_or_inf = 0;
		rc = report( ctx, "PV::convert_to_audio", flan_b200_convert_to_audio( ctx, reinterpret_cast<const float *>( d_pv ),
			get_num_channels(), get_num_frames(), get_num_bins(), get_sample_rate(), get_analysis_rate(), get_window_size(),
			d_audio, &cancel.value, &nan_or_inf ) );
		if( nan_or_inf )                                                     // AudioPV.cpp:88-89: warn and carry on
			std::cout << "flan::convert_to_audio recieved a nan or infinite value. This often happens when dividing by zero in an earlier algorithm.";
		}
	if( rc != FLAN_B200_OK || canceller ) return Audio::create_null();
	return Audio( AudioBuffer::from_device_result( af, std::move( data ) ) );
	}

Audio PV::convert_to_lr_audio( flan_CANCEL_ARG_CPP ) const
	{
	if( get_num_channels() != 2 ) return Audio::create_null();           // AudioPV.cpp:143
	return convert_to_audio( canceller ).convert_to_left_right();
	}

}
