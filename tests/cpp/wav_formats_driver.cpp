// tests/cpp/wav_formats_driver.cpp -- user code that loads and saves WAV files of several sample types through the
// reference's C++ API, with libsndfile's format names (SF_FORMAT_WAV | SF_FORMAT_PCM_16 ...) written unqualified as
// code against the reference writes them. Exposed through extern "C" for pytest.
#include "flan/Audio/Audio.h"

#include <cstring>

using namespace flan;

extern "C" {

// The libsndfile format a test names: 0 = save( path ) with the default format, 1 = WAV | FLOAT, 2 = WAV | PCM_16,
// 3 = WAV | PCM_24, 4 = AIFF | PCM_16, 5 = WAV | PCM_S8, 6 = WAV | PCM_16 | big-endian, 7 = WAV | PCM_U8 | little-endian,
// 8 = WAV | PCM_32 | file endianness, 9 = WAV | DOUBLE.
int api_wav_save( const float * audio, int C, int n, float sr, const char * path, int which )
	{
	Audio a = Audio::create_from_buffer( std::vector<float>( audio, audio + size_t( C ) * n ), C, sr );
	bool ok = false;
	switch( which )
		{
		case 0: ok = a.save( path ); break;
		case 1: ok = a.save( path, SF_FORMAT_WAV | SF_FORMAT_FLOAT ); break;
		case 2: ok = a.save( path, SF_FORMAT_WAV | SF_FORMAT_PCM_16 ); break;
		case 3: ok = a.save( path, SF_FORMAT_WAV | SF_FORMAT_PCM_24 ); break;
		case 4: ok = a.save( path, SF_FORMAT_AIFF | SF_FORMAT_PCM_16 ); break;
		case 5: ok = a.save( path, SF_FORMAT_WAV | SF_FORMAT_PCM_S8 ); break;
		case 6: ok = a.save( path, SF_FORMAT_WAV | SF_FORMAT_PCM_16 | SF_ENDIAN_BIG ); break;
		case 7: ok = a.save( path, SF_FORMAT_WAV | SF_FORMAT_PCM_U8 | SF_ENDIAN_LITTLE ); break;
		case 8: ok = a.save( path, SF_FORMAT_WAV | SF_FORMAT_PCM_32 | SF_ENDIAN_FILE ); break;
		case 9: ok = a.save( path, SF_FORMAT_WAV | SF_FORMAT_DOUBLE ); break;
		default: return -1;
		}
	return ok ? 1 : 0;
	}

// Loads a WAV file; returns its frame count (and channels, sample rate, up to `capacity` samples), or -1.
int api_wav_load( const char * path, float * audio_out, int64_t capacity, int * C_out, float * sr_out )
	{
	Audio a;
	if( !a.load( path ) ) return -1;
	*C_out = a.get_num_channels();
	*sr_out = float( a.get_sample_rate() );
	const size_t count = a.get_buffer().size();
	if( int64_t( count ) > capacity ) return -1;
	std::memcpy( audio_out, a.get_buffer().data(), sizeof( float ) * count );
	return a.get_num_frames();
	}

}
