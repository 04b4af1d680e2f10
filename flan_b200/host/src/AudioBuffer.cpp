// flan::AudioBuffer of the B200 build (surface of reference src/flan/Audio/AudioBuffer.{h,cpp}; own implementation).
#include "flan/Audio/AudioBuffer.h"

#include <algorithm>
#include <cmath>
#include <iostream>
#include <ostream>

#include "flan_b200.h"

namespace flan {

AudioBuffer::AudioBuffer() : format(), buffer() {}

AudioBuffer::AudioBuffer( std::vector<float> && data, Channel num_channels, FrameRate sr )
	: format(), buffer()
	{
	format.num_channels = num_channels;
	format.num_frames = num_channels > 0 ? Frame( data.size() / size_t( num_channels ) ) : 0;
	format.sample_rate = sr;
	buffer = b200::Mirror<Sample>( std::move( data ) );
	}

AudioBuffer::AudioBuffer( const Format & f )
	: format( f )
	, buffer( size_t( std::max( f.num_channels, 0 ) ) * size_t( std::max( f.num_frames, 0 ) ) )
	{}

AudioBuffer AudioBuffer::from_device_result( const Format & f, b200::Mirror<Sample> && data )
	{
	AudioBuffer out;
	out.format = f;
	out.buffer = std::move( data );
	return out;
	}

AudioBuffer AudioBuffer::copy() const
	{
	AudioBuffer out;
	out.format = format;
	out.buffer = buffer.deep_copy();
	return out;
	}

bool AudioBuffer::is_null() const { return buffer.empty() || get_sample_rate() == 0; }

bool AudioBuffer::is_nan_or_inf() const
	{
	for( Sample s : buffer.host() )
		if( std::isnan( s ) || std::isinf( s ) ) return true;
	return false;
	}

void AudioBuffer::print_summary() const { std::cout << *this; }

Sample AudioBuffer::get_sample( Channel c, Frame f ) const { return buffer.host()[get_buffer_pos( c, f )]; }
AudioBuffer::Format AudioBuffer::get_format() const { return format; }
Channel AudioBuffer::get_num_channels() const { return format.num_channels; }
Frame AudioBuffer::get_num_frames() const { return format.num_frames; }
FrameRate AudioBuffer::get_sample_rate() const { return format.sample_rate; }
Second AudioBuffer::frame_to_time( fFrame f ) const { return f / get_sample_rate(); }
fFrame AudioBuffer::time_to_frame( Second t ) const { return t * float( get_sample_rate() ); }
Second AudioBuffer::get_length() const { return frame_to_time( get_num_frames() ); }

Sample AudioBuffer::get_max_sample_magnitude( Second start_time, Second end_time ) const
	{
	if( end_time == 0 ) end_time = get_length();
	const Frame lo = std::clamp( Frame( time_to_frame( start_time ) ), 0, get_num_frames() - 1 );
	const Frame hi = std::clamp( Frame( time_to_frame( end_time ) ), 0, get_num_frames() - 1 );
	const std::vector<Sample> & h = buffer.host();
	Sample m = 0;
	for( Channel c = 0; c < get_num_channels(); ++c )
		for( Frame f = lo; f < hi; ++f )
			m = std::max( m, std::abs( h[get_buffer_pos( c, f )] ) );
	return m;
	}

void AudioBuffer::set_sample( Channel c, Frame f, Sample s ) { buffer.host_mut()[get_buffer_pos( c, f )] = s; }
Sample & AudioBuffer::get_sample( Channel c, Frame f ) { return buffer.host_mut()[get_buffer_pos( c, f )]; }

void AudioBuffer::clear_buffer()
	{
	std::vector<Sample> & h = buffer.host_mut();
	std::fill( h.begin(), h.end(), 0.0f );
	}

Sample * AudioBuffer::get_sample_pointer( Channel c, Frame f ) { return buffer.host_mut().data() + get_buffer_pos( c, f ); }
const Sample * AudioBuffer::get_sample_pointer( Channel c, Frame f ) const { return buffer.host().data() + get_buffer_pos( c, f ); }
std::vector<Sample> & AudioBuffer::get_buffer() { return buffer.host_mut(); }
const std::vector<Sample> & AudioBuffer::get_buffer() const { return buffer.host(); }

std::vector<Sample>::const_iterator AudioBuffer::channel_begin( Channel c ) const { return buffer.host().begin() + get_buffer_pos( c, 0 ); }
std::vector<Sample>::const_iterator AudioBuffer::channel_end( Channel c ) const { return buffer.host().begin() + get_buffer_pos( c + 1, 0 ); }

size_t AudioBuffer::get_buffer_pos( Channel c, Frame f ) const
	{
	return size_t( c ) * size_t( get_num_frames() ) + size_t( f );
	}

std::ostream & operator<<( std::ostream & os, const AudioBuffer & a )
	{
	os << "\n=========================== AudioBuffer Info ==========================="
	   << "\nChannels:\t" << a.get_num_channels()
	   << "\nFrames:\t\t" << a.get_num_frames()
	   << "\nSample Rate:\t" << a.get_sample_rate()
	   << "\nLength:\t\t" << a.get_length() << " seconds"
	   << "\n========================================================================\n\n";
	return os;
	}


// ---- WAV files (reference AudioBuffer.cpp:80-192 through libsndfile): the sample codecs run on the GPU ---------------

static_assert( SF_FORMAT_PCM_U8 == FLAN_B200_WAV_PCM_U8 && SF_FORMAT_PCM_16 == FLAN_B200_WAV_PCM_16 &&
               SF_FORMAT_PCM_24 == FLAN_B200_WAV_PCM_24 && SF_FORMAT_PCM_32 == FLAN_B200_WAV_PCM_32 &&
               SF_FORMAT_FLOAT == FLAN_B200_WAV_FLOAT && SF_FORMAT_DOUBLE == FLAN_B200_WAV_DOUBLE, "libsndfile's sub-type codes" );

// The FLAN_B200_WAV_* sample type a libsndfile format asks for, or 0 where this build does not write it: another major
// format, big-endian, or a sub-type libsndfile does not accept for WAV (PCM_S8) or this build does not know.
static int wav_subtype_of( int file_format )
	{
	if( file_format == -1 ) return FLAN_B200_WAV_PCM_24;                  // AudioBuffer.cpp:136
	if( ( file_format & SF_FORMAT_TYPEMASK ) != SF_FORMAT_WAV ) return 0;
	const int endian = file_format & SF_FORMAT_ENDMASK;
	if( endian != SF_ENDIAN_FILE && endian != SF_ENDIAN_LITTLE ) return 0;
	if( file_format & ~( SF_FORMAT_TYPEMASK | SF_FORMAT_SUBMASK | SF_FORMAT_ENDMASK ) ) return 0;
	switch( file_format & SF_FORMAT_SUBMASK )          // libsndfile's sub-type codes are the FLAN_B200_WAV_* codes
		{
		case SF_FORMAT_PCM_U8: case SF_FORMAT_PCM_16: case SF_FORMAT_PCM_24: case SF_FORMAT_PCM_32:
		case SF_FORMAT_FLOAT: case SF_FORMAT_DOUBLE:
			return file_format & SF_FORMAT_SUBMASK;
		default: return 0;
		}
	}

bool AudioBuffer::save( const std::string & filename, int file_format ) const
	{
	const int subtype = wav_subtype_of( file_format );
	if( !subtype )
		{
		std::cout << "Sound file formatting invalid while attempting to save to " << filename << ",\n"
		          << "(the B200 build writes WAV, little-endian, with PCM_U8, PCM_16, PCM_24, PCM_32, FLOAT or DOUBLE samples)" << std::endl;
		return false;
		}
	flan_b200_ctx * ctx = b200::context();
	if( !ctx ) return false;
	const Sample * d = buffer.empty() ? nullptr : buffer.device();
	if( !buffer.empty() && !d ) return false;
	const int rc = flan_b200_save_wav_as( ctx, filename.c_str(), d, get_num_channels(), get_num_frames(), get_sample_rate(), subtype );
	if( rc != FLAN_B200_OK ) std::cout << flan_b200_last_error( ctx ) << std::endl;
	return rc == FLAN_B200_OK;
	}

bool AudioBuffer::load( const std::string & filename )
	{
	flan_b200_ctx * ctx = b200::context();
	if( !ctx ) return false;
	int C = 0; int64_t n = 0; float sr = 0;
	if( flan_b200_wav_info( ctx, filename.c_str(), &C, &n, &sr ) != FLAN_B200_OK )
		{
		std::cout << filename << " could not be opened: " << flan_b200_last_error( ctx ) << std::endl;     // AudioBuffer.cpp:88-92
		return false;
		}
	Format f;
	f.num_channels = C; f.num_frames = Frame( n ); f.sample_rate = sr;   // AudioBuffer.cpp:95-97
	Sample * d = nullptr;
	b200::Mirror<Sample> data = b200::Mirror<Sample>::device_result( size_t( C ) * size_t( n ), &d );
	if( !d ) return false;
	if( flan_b200_load_wav( ctx, filename.c_str(), d, int64_t( C ) * n ) != FLAN_B200_OK )
		{
		std::cout << flan_b200_last_error( ctx ) << std::endl;
		return false;
		}
	*this = from_device_result( f, std::move( data ) );
	return true;
	}

}
