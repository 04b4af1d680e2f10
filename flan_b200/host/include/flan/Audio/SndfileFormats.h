// libsndfile's format names for AudioBuffer::save( filename, format ), so that code written against the reference
// (SF_FORMAT_WAV | SF_FORMAT_PCM_16 ...) compiles unchanged. Where libsndfile's own header is present it is used, so a
// program that also includes it sees each name once; otherwise the names are declared here with libsndfile's values.
#pragma once

#if __has_include( <sndfile.h> )
#include <sndfile.h>
#else
enum
	{
	// major formats
	SF_FORMAT_WAV = 0x010000,
	SF_FORMAT_AIFF = 0x020000,

	// sub-types
	SF_FORMAT_PCM_S8 = 0x0001,
	SF_FORMAT_PCM_16 = 0x0002,
	SF_FORMAT_PCM_24 = 0x0003,
	SF_FORMAT_PCM_32 = 0x0004,
	SF_FORMAT_PCM_U8 = 0x0005,
	SF_FORMAT_FLOAT = 0x0006,
	SF_FORMAT_DOUBLE = 0x0007,

	// endianness
	SF_ENDIAN_FILE = 0x00000000,
	SF_ENDIAN_LITTLE = 0x10000000,
	SF_ENDIAN_BIG = 0x20000000,

	SF_FORMAT_SUBMASK = 0x0000FFFF,
	SF_FORMAT_TYPEMASK = 0x0FFF0000,
	SF_FORMAT_ENDMASK = 0x30000000
	};
#endif
