// flan::AudioBuffer of the B200 build: the reference's public surface (src/flan/Audio/AudioBuffer.h:20-228) for
// everything on the phase-vocoder path, over device-resident storage (flan/b200_storage.h). Layout contract:
// planar, channel-major, pos = channel * num_frames + frame (AudioBuffer.cpp:479-482) -- computed in 64 bits here.
// File I/O: WAV with libsndfile's sample types for it (8-bit unsigned, 16-, 24- and 32-bit PCM, 32- and 64-bit float;
// 24-bit PCM is the reference's default save format, AudioBuffer.cpp:136), with the sample conversion and the
// (de)interleave on the GPU; libsndfile's other major formats and its metadata strings are outside the scope of this build.
#pragma once

#include <iosfwd>
#include <string>
#include <vector>

#include "flan/defines.h"
#include "flan/b200_storage.h"
#include "flan/Audio/SndfileFormats.h"

namespace flan {

class AudioBuffer
{
public:
	AudioBuffer( const AudioBuffer & ) = delete;
	AudioBuffer( AudioBuffer && ) = default;
	AudioBuffer & operator=( const AudioBuffer & ) = delete;
	AudioBuffer & operator=( AudioBuffer && ) = default;
	~AudioBuffer() = default;

	struct Format
		{
		Channel num_channels = 0;
		Frame num_frames = 0;
		FrameRate sample_rate = 48000;
		};

	AudioBuffer();
	AudioBuffer( std::vector<float> && buffer, Channel num_channels, FrameRate = 48000 );
	AudioBuffer( const Format & format );      // zero-filled, like the reference (AudioBuffer.cpp:26-29)

	AudioBuffer copy() const;
	bool is_null() const;
	bool is_nan_or_inf() const;
	void print_summary() const;

	Sample get_sample( Channel channel, Frame frame ) const;
	Format get_format() const;
	Channel get_num_channels() const;
	Frame get_num_frames() const;
	FrameRate get_sample_rate() const;
	Second get_length() const;
	Sample get_max_sample_magnitude( Second start_time = 0, Second end_time = 0 ) const;
	Second frame_to_time( fFrame ) const;
	fFrame time_to_frame( Second ) const;

	void set_sample( Channel channel, Frame frame, Sample sample );
	Sample & get_sample( Channel channel, Frame frame );
	void clear_buffer();
	Sample * get_sample_pointer( Channel channel, Frame frame );
	const Sample * get_sample_pointer( Channel channel, Frame frame ) const;
	std::vector<Sample> & get_buffer();
	const std::vector<Sample> & get_buffer() const;
	std::vector<Sample>::const_iterator channel_begin( Channel channel ) const;
	std::vector<Sample>::const_iterator channel_end( Channel channel ) const;
	size_t get_buffer_pos( Channel, Frame ) const;

	// B200 build: device-side view for the conversion entry points (not part of the reference's surface)
	/** Load a WAV file of PCM (8, 16, 24, 32 bits) or float (32, 64 bits) samples (reference AudioBuffer::load,
	 *  AudioBuffer.cpp:80-128). false + message on failure. */
	bool load( const std::string & filename );
	/** Save as WAV, samples clamped to [-1,1] (reference AudioBuffer::save, AudioBuffer.cpp:130-170). \param format is
	 *  libsndfile's: -1 (the default, 24-bit PCM) or SF_FORMAT_WAV | SF_FORMAT_PCM_U8 / _PCM_16 / _PCM_24 / _PCM_32 /
	 *  _FLOAT / _DOUBLE, with SF_ENDIAN_FILE or SF_ENDIAN_LITTLE. Any other format prints a message and returns false. */
	bool save( const std::string & filename, int format = -1 ) const;

	const b200::Mirror<Sample> & storage() const { return buffer; }
	static AudioBuffer from_device_result( const Format & format, b200::Mirror<Sample> && data );

private:
	Format format;
	b200::Mirror<Sample> buffer;
};

std::ostream & operator<<( std::ostream & os, const AudioBuffer & audio );

}
